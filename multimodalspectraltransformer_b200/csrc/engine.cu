// C-ABI entry points of the MMT B200 engine (include/mmt_b200.h) and the host-side
// drivers that sequence the kernels for encode / decode.
#include "engine.cuh"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_decode.cuh"
#include "kernels_ffn.cuh"
#include "kernels_attn5.cuh"
#include "kernels_compact.cuh"
#include "kernels_beam.cuh"
#include "kernels_sbs.cuh"
#include "kernels_smiles.cuh"
#include "kernels_retire.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>

namespace mmt {
thread_local std::string g_last_error;

static const char* kEmbedKeys[5] = {
    "linear_spec_embedding_1H.point_embedding_layer_1H.fc_H",
    "linear_spec_embedding_13C.point_embedding_layer_13C.fc_C",
    "linear_spec_embedding_HSQC.point_embedding_layer_HSQC.fc_HSQC",
    "linear_spec_embedding_COSY.point_embedding_layer_COSY.fc_COSY",
    "linear_spec_embedding_IR.linear_spec_embedding_IR"};
static const char* kEncNames[6] = {"encoder_1H", "encoder_13C", "encoder_HSQC", "encoder_COSY", "encoder_IR", "encoder_cross"};

// Every kernel launch goes through prof_pre()/check_launch(): counts launches and, when
// profiling is enabled (mmt_profile_enable), brackets the launch with CUDA events recorded
// on the launching stream so bench.py can report per-kernel-class device time.
static void prof_pre(mmt_engine* e, cudaStream_t s) {
    if (!e->profiling) return;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    cudaEventRecord(a, s);
    e->prof_open = {a, b};
}
static int check_launch(mmt_engine* e, const char* what, cudaStream_t s = nullptr, double work = 0.0) {
    e->launches++;
    cudaError_t err = cudaGetLastError();
    if (e->profiling && e->prof_open.first) {
        cudaEventRecord(e->prof_open.second, s);
        e->prof_records.push_back({what, e->prof_open.first, e->prof_open.second, work});
        e->prof_open = {nullptr, nullptr};
    }
    if (err != cudaSuccess) MMT_FAIL(std::string(what) + " launch -> " + cudaGetErrorString(err));
    return 0;
}

// Launch with (optionally) the programmatic-dependent-launch attribute: the kernel may be scheduled while its
// predecessor in the stream drains; it synchronises on the predecessor itself with griddepcontrol.wait
// (common.cuh pdl_wait).  Captured into the decode-step graph as a programmatic dependency edge.
template <typename P>
static void launch_kernel(void (*kernel)(P), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, const P& params) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, params);     // errors surface through cudaGetLastError() in check_launch
}

// the same as a thread-block-cluster launch (cluster_x CTAs along x; grid.x must be a multiple of it)
template <typename P>
static void launch_kernel_cluster(void (*kernel)(P), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, unsigned cluster_x, const P& params) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cluster_x; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 2 : 1;
    cudaLaunchKernelEx(&cfg, kernel, params);
}

// the same for kernels that take their arguments one by one
template <typename... KArgs, typename... Args>
static void launch_args(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Scope of one C-ABI call on an engine: serialises the host side (the arena, the pinned staging buffer, the graph cache and
// the launch counter are per engine) and orders the device side across streams -- a call on another stream than the
// previous call's first waits for the event that call recorded at its end, so the shared workspace is never aliased by
// two streams' work.  Calls on the same stream are ordered by the stream itself.
struct EngineCall {
    mmt_engine* e; cudaStream_t s; std::unique_lock<std::mutex> lk;
    EngineCall(mmt_engine* e_, cudaStream_t s_) : e(e_), s(s_), lk(e_->mu) {
        cudaSetDevice(e->device);
        if (e->last_use_valid && e->last_stream != s) cudaStreamWaitEvent(s, e->last_use, 0);
    }
    ~EngineCall() {
        if (!e->last_use && cudaEventCreateWithFlags(&e->last_use, cudaEventDisableTiming) != cudaSuccess) { e->last_use = nullptr; cudaGetLastError(); return; }
        if (cudaEventRecord(e->last_use, s) == cudaSuccess) { e->last_use_valid = true; e->last_stream = s; }
        else { e->last_use_valid = false; cudaGetLastError(); }
    }
};

static int ensure_arena(mmt_engine* e, size_t bytes) {
    if (bytes <= e->arena_bytes) return 0;
    if (e->arena) {
        MMT_CUDA(cudaDeviceSynchronize());
        MMT_CUDA(cudaFree(e->arena)); e->arena = nullptr; e->arena_bytes = 0;
    }
    size_t want = bytes + (bytes >> 3);
    MMT_CUDA(cudaMalloc(&e->arena, want));
    e->arena_bytes = want;
    return 0;
}

// A call's workspace in the arena: `plan` lays out its buffers with ar.get, once to measure them, and -- after the arena
// has grown to fit -- once more to place them.
template <typename F>
static int plan_arena(mmt_engine* e, Arena& ar, F&& plan) {
    ar = Arena();
    plan();
    MMT_TRY(ensure_arena(e, ar.off));
    ar.plan = false; ar.base = e->arena; ar.cap = e->arena_bytes; ar.off = 0;
    plan();
    return 0;
}

// torch's Philox launch geometry for a draw of `numel` elements, on the call's device description (sm_count /
// max_threads_per_sm > 0) or the engine's device; *inc = the generator advance of one such draw
static RngGeom rng_geom(const mmt_engine* e, uint64_t seed, uint64_t offset, int64_t numel, int sm_count, int max_threads_per_sm,
                        uint64_t* inc) {
    const int smc = sm_count > 0 ? sm_count : e->sm_count;
    const int mts = max_threads_per_sm > 0 ? max_threads_per_sm : e->max_threads_per_sm;
    RngGeom g;
    g.seed = seed; g.offset = offset; g.numel = numel; g.threads = torch_rng_threads(numel, smc, mts);
    *inc = torch_rng_increment(numel, smc, mts);
    return g;
}

// ---------------------------------------------------------------------------
// launch helpers
// ---------------------------------------------------------------------------
// tile_rows > 0 picks the tile shape for that many rows instead of maxM (a compacted decode wave keeps the shape of its
// starting size: the two shapes need not round alike)
static int launch_gemm(mmt_engine* e, GemmParams& p, int ngroups, int maxM, cudaStream_t s, int64_t tile_rows = 0) {
    if (maxM <= 0) return 0;
    if (p.splits < 1) p.splits = 1;
    if ((tile_rows > 0 ? tile_rows : maxM) >= 1024) {
        dim3 grid((p.N + 127) / 128, (maxM + 127) / 128, ngroups * p.splits);
        prof_pre(e, s);
        gemm_nt_f32<128, 128, 8, 8><<<grid, 256, 0, s>>>(p);
    } else {
        dim3 grid((p.N + 63) / 64, (maxM + 31) / 32, ngroups * p.splits);
        prof_pre(e, s);
        gemm_nt_f32<32, 64, 2, 4><<<grid, 256, 0, s>>>(p);
    }
    double rows = 0;
    for (int i = 0; i < ngroups; ++i) rows += p.g[i].M;
    return check_launch(e, "gemm_nt_f32", s, 2.0 * rows * p.N * p.K);
}

static GemmParams gemm_params(int N, int K, int64_t ldc, int act) {
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.N = N; p.K = K; p.ldc = ldc; p.act = act; p.splits = 1; p.out_mode = GEMM_OUT_ROWMAJOR;
    return p;
}

static int pick_splits(int M, int N, int K) {
    if (M >= 1024) return 1;
    int tiles = ((M + 31) / 32) * ((N + 63) / 64);
    int s = 1;
    while (s < 16 && tiles * s < 256 && (K / (s * 2)) >= 64) s *= 2;
    return s;
}

static int launch_ln(mmt_engine* e, LnParams& p, int ngroups, int maxM, cudaStream_t s) {
    if (maxM <= 0) return 0;
    dim3 grid((maxM + 7) / 8, ngroups);
    prof_pre(e, s);
    bias_res_layernorm<<<grid, 256, 0, s>>>(p);
    return check_launch(e, "bias_res_layernorm", s);
}

// ---------------------------------------------------------------------------
// tcgen05 GEMM launch (bf16 operands): tensor maps are encoded on the host per call
// ---------------------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_tmapEncodeTiled g_encode_tiled = nullptr;

static int tc_init(mmt_engine* e) {
    if (e->tc_ready) return 0;
    if (!g_encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        MMT_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) MMT_FAIL("cuTensorMapEncodeTiled not available from the driver");
        g_encode_tiled = (PFN_tmapEncodeTiled)fn;
    }
    const int max_smem = TC_MAX_STAGES * TC_STAGE_BYTES_WSPLIT + 1024;
    MMT_CUDA(cudaFuncSetAttribute(gemm_bf16_tc<TC_EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    MMT_CUDA(cudaFuncSetAttribute(gemm_bf16_tc<TC_EPI_LN>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
    MMT_CUDA(cudaFuncSetAttribute(attn_encoder_tc5, cudaFuncAttributeMaxDynamicSharedMemorySize, A5_SMEM_BYTES));
    MMT_CUDA(cudaFuncSetAttribute(ffn_fused_tc<TC_EPI_STORE, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff_smem_bytes<1>()));
    MMT_CUDA(cudaFuncSetAttribute(ffn_fused_tc<TC_EPI_LN, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff_smem_bytes<1>()));
    MMT_CUDA(cudaFuncSetAttribute(ffn_fused_tc<TC_EPI_STORE, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff_smem_bytes<0>()));
    MMT_CUDA(cudaFuncSetAttribute(ffn_fused_tc<TC_EPI_LN, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff_smem_bytes<0>()));
    MMT_CUDA(cudaFuncSetAttribute(ffn_fused_tc<TC_EPI_LN, 0, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, ff_smem_bytes<0, 1>()));
    e->tc_ready = true;
    return 0;
}

// [rows, cols] bf16 matrix, `ld` elements between rows; box = 64 (K) x 128 (rows), 128-byte swizzle
static int make_tmap(CUtensorMap* m, const __nv_bfloat16* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows = TC_BM) {
    if (((uintptr_t)ptr & 15) || (ld * 2) % 16) MMT_FAIL("tensor map: operand must be 16-byte aligned with a 16-byte multiple row pitch");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) MMT_FAIL("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)r));
    return 0;
}

static TcGemmParams tc_params(int M, int N, int K) {
    TcGemmParams p;
    memset(&p, 0, sizeof(p));
    p.M = M; p.N = N; p.K = K; p.splits = 1; p.eps = 1e-5f;
    p.S_in = M > 0 ? M : 1; p.stride_b = 0; p.stride_s = 1; p.off = 0;
    return p;
}

// sample_tokens over sp.N rows (sample_tokens<true> with per-column controls).  `plan_rows` fixes the variant: a decode
// wave's starting size (a compacted wave keeps it), else N.
static int launch_sample(mmt_engine* e, SampleParams& sp, int64_t plan_rows, bool controlled, bool pdl, cudaStream_t s) {
    if (!e->sample_ready) {   // fc_out sits in dynamic shared memory (33 KB at the 64-row maximum, next to 20 KB of static row buffers)
        MMT_CUDA(cudaFuncSetAttribute(sample_tokens<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sample_smem_bytes(VOCAB_MAX)));
        MMT_CUDA(cudaFuncSetAttribute(sample_tokens<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sample_smem_bytes(VOCAB_MAX)));
        e->sample_ready = true;
    }
    // rows per CTA and pass: 2 when the input is still spread over FFN2 partials, else 8 warps' rows; at most four resident
    // waves of CTAs.  Small waves take one row per warp (latency), large ones four (shared-memory traffic).
    sp.rows_per_warp = plan_rows >= 8192 ? SAMPLE_NR : 1;
    const int rpc = sp.part ? 2 : 8 * sp.rows_per_warp;
    const int64_t groups = (sp.N + rpc - 1) / rpc;
    prof_pre(e, s);
    launch_kernel(controlled ? sample_tokens<true> : sample_tokens<false>, dim3((unsigned)std::min<int64_t>(groups, (int64_t)e->sm_count * 4)),
                  dim3(256), sample_smem_bytes(sp.V), s, pdl, sp);
    return check_launch(e, controlled ? "sample_tokens_controlled" : "sample_tokens", s);
}

// A [M,K] bf16 (row pitch lda), W [N,K] bf16 (dense), optional low-order weight term Wlo; the
// rest of `p` is filled by the caller
struct TcChain { const __nv_bfloat16 *W, *Wlo; const float* bias; float* out; int64_t ld; };
static int launch_tc(mmt_engine* e, TcGemmParams& p, const __nv_bfloat16* A, int64_t lda, const __nv_bfloat16* W, int epi, cudaStream_t s,
                     const __nv_bfloat16* Wlo = nullptr, bool pdl = false, const TcChain* chain = nullptr) {
    if (p.M <= 0) return 0;
    MMT_TRY(tc_init(e));
    if (p.K % TC_BK || p.N % 4) MMT_FAIL("tcgen05 GEMM needs K % 64 == 0 and N % 4 == 0");
    if (epi == TC_EPI_LN && (p.N != D || p.splits != 1)) MMT_FAIL("LayerNorm epilogue needs N == 128 and no split-K");
    const int kb_total = p.K / TC_BK;
    if (p.splits < 1) p.splits = 1;
    if (p.splits > kb_total) p.splits = kb_total;
    const int kb_per = (kb_total + p.splits - 1) / p.splits;
    p.splits = (kb_total + kb_per - 1) / kb_per;          // no empty split
    p.wsplit = Wlo != nullptr;
    p.stages = std::min(kb_per, (kb_per > 2 && !p.wsplit) ? 3 : 2);
    MMT_TRY(make_tmap(&p.tmA, A, p.M, p.K, lda));
    MMT_TRY(make_tmap(&p.tmW, W, p.N, p.K, p.K));
    if (p.wsplit) MMT_TRY(make_tmap(&p.tmW2, Wlo, p.N, p.K, p.K));
    size_t smem = (size_t)std::max(p.stages * (p.wsplit ? TC_STAGE_BYTES_WSPLIT : TC_STAGE_BYTES), TC_STAGING_BYTES) + 1024;
    if (chain) {
        if (epi != TC_EPI_LN || !chain->W || !chain->bias || !chain->out) MMT_FAIL("chained projection needs the LayerNorm epilogue and a weight");
        p.chain = chain->Wlo ? 2 : 1; p.chain_bias = chain->bias; p.chain_out = chain->out; p.ld_chain = chain->ld;
        MMT_TRY(make_tmap(&p.tmC, chain->W, D, D, D));
        if (chain->Wlo) MMT_TRY(make_tmap(&p.tmC2, chain->Wlo, D, D, D));
        smem = ((smem - 1024 + 1023) & ~size_t(1023)) + (chain->Wlo ? TC_CHAIN_BYTES : TC_CHAIN_BYTES - 2 * TC_SLAB_BYTES) + 1024;
    }
    dim3 grid((p.N + TC_BN - 1) / TC_BN, (p.M + TC_BM - 1) / TC_BM, p.splits);
    prof_pre(e, s);
    if (epi == TC_EPI_LN) launch_kernel(gemm_bf16_tc<TC_EPI_LN>, grid, dim3(TC_THREADS), smem, s, pdl, p);
    else launch_kernel(gemm_bf16_tc<TC_EPI_STORE>, grid, dim3(TC_THREADS), smem, s, pdl, p);
    return check_launch(e, epi == TC_EPI_LN ? "gemm_bf16_tc_ln" : "gemm_bf16_tc", s, 2.0 * p.M * p.N * p.K);
}

static FfnParams ffn_params(int M, int F) {
    FfnParams p;
    memset(&p, 0, sizeof(p));
    p.M = M; p.N = D; p.F = F; p.splits = 1; p.eps = 1e-5f; p.ld_f32 = D; p.ld_b16 = D;
    p.S_in = M > 0 ? M : 1; p.stride_b = 0; p.stride_s = 1; p.off = 0;
    return p;
}

// Fused FFN (kernels_ffn.cuh): X [M,128] bf16 (row pitch ldx); W1 [F,128] / W2 [128,F] as bf16 hi (+ lo) terms.
// splits == 1 with epi == TC_EPI_LN: out = LN(res + b2 + FFN(X)); splits > 1: raw partials to out_f32.
struct FfnPro { const __nv_bfloat16 *W, *Wlo; const float *bias, *gamma, *beta; float* out; };
static int launch_ffn(mmt_engine* e, FfnParams& p, const __nv_bfloat16* X, int64_t ldx, const __nv_bfloat16* W1, const __nv_bfloat16* W1lo,
                      const __nv_bfloat16* W2, const __nv_bfloat16* W2lo, int epi, cudaStream_t s, bool pdl = false, const FfnPro* pro = nullptr) {
    if (p.M <= 0) return 0;
    MMT_TRY(tc_init(e));
    if (p.F % FF_CH || p.F > FF_MAX_F || p.F < FF_CH) MMT_FAIL("fused FFN needs d_ff % 64 == 0 and d_ff <= 2048");
    const int chunks = p.F / FF_CH;
    if (p.splits < 1) p.splits = 1;
    while (chunks % p.splits) --p.splits;
    if (epi == TC_EPI_LN && p.splits != 1) MMT_FAIL("fused FFN: the LayerNorm epilogue needs splits == 1");
    p.wsplit = (W1lo && W2lo) ? 1 : 0;
    MMT_TRY(make_tmap(&p.tmX, X, p.M, D, ldx));
    MMT_TRY(make_tmap(&p.tmW1, W1, p.F, D, D, FF_CH));
    MMT_TRY(make_tmap(&p.tmW2, W2, D, p.F, p.F));
    if (p.wsplit) {
        MMT_TRY(make_tmap(&p.tmW1lo, W1lo, p.F, D, D, FF_CH));
        MMT_TRY(make_tmap(&p.tmW2lo, W2lo, D, p.F, p.F));
    }
    if (pro) {
        if (epi != TC_EPI_LN || p.splits != 1 || !pro->W || !pro->out || p.res != pro->out)
            MMT_FAIL("fused FFN prologue needs the LayerNorm epilogue, a weight and the residual buffer as its output");
        p.pro = pro->Wlo ? 2 : 1; p.pro_bias = pro->bias; p.pro_gamma = pro->gamma; p.pro_beta = pro->beta; p.pro_out = pro->out;
        MMT_TRY(make_tmap(&p.tmP, pro->W, D, D, D));
        if (pro->Wlo) MMT_TRY(make_tmap(&p.tmPlo, pro->Wlo, D, D, D));
    }
    dim3 grid(p.splits, (p.M + TC_BM - 1) / TC_BM);
    if (const char* v = getenv("MMT_FFN_KNOCK")) p.knock = atoi(v);
    prof_pre(e, s);
    if (p.wsplit) {
        if (epi == TC_EPI_LN) launch_kernel(ffn_fused_tc<TC_EPI_LN, 1>, grid, dim3(FF_THREADS), ff_smem_bytes<1>(), s, pdl, p);
        else launch_kernel(ffn_fused_tc<TC_EPI_STORE, 1>, grid, dim3(FF_THREADS), ff_smem_bytes<1>(), s, pdl, p);
    } else {   // hi term only: the deeper pipeline variant
        if (epi == TC_EPI_LN && p.splits == 1 && p.F % (2 * FF_CH) == 0 && e->use_ffn_wide)      // 128-column chunks
            launch_kernel(ffn_fused_tc<TC_EPI_LN, 0, 1>, grid, dim3(ff_threads<0, 1>()), ff_smem_bytes<0, 1>(), s, pdl, p);
        else if (epi == TC_EPI_LN) launch_kernel(ffn_fused_tc<TC_EPI_LN, 0>, grid, dim3(FF_THREADS), ff_smem_bytes<0>(), s, pdl, p);
        else launch_kernel(ffn_fused_tc<TC_EPI_STORE, 0>, grid, dim3(FF_THREADS), ff_smem_bytes<0>(), s, pdl, p);
    }
    return check_launch(e, "ffn_fused_tc", s, 4.0 * p.M * D * p.F);
}

// ---------------------------------------------------------------------------
// encoder
// ---------------------------------------------------------------------------
struct ModeLayout {
    int present[5];
    int S_m[5];      // sequence length of each block in the concatenated memory
    int n_x[5];
    int off[5];
    int S_total;
    int float_mask;
    int has_MF, has_MS, has_MW;
};

static ModeLayout mode_layout(const mmt_model_desc& d, uint32_t mode) {
    ModeLayout L;
    memset(&L, 0, sizeof(L));
    L.has_MF = (mode & MMT_MODE_MF) != 0; L.has_MS = (mode & MMT_MODE_MS) != 0; L.has_MW = (mode & MMT_MODE_MW) != 0;
    const int P = d.pad_points;
    const int extra = (L.has_MF ? P : 0) + (L.has_MS ? P : 0) + (L.has_MW ? 1 : 0);
    const int fdim = L.has_MS ? 193 : 129, fdim_ir = L.has_MS ? 130 : 66;   // models_MMT_v15_4.py:834-835
    int off = 0;
    for (int m = 0; m < 5; ++m) {
        L.present[m] = (mode >> m) & 1;
        L.n_x[m] = (m == 4) ? 1 : P;
        if (L.present[m]) L.S_m[m] = L.n_x[m] + extra;
        else L.S_m[m] = (m == 3) ? 65 : (m == 4 ? fdim_ir : fdim);             // :852, :912, :933
        L.off[m] = off;
        off += L.S_m[m];
        if (m < 4 && !L.present[m]) L.float_mask = 1;
    }
    L.S_total = off;
    return L;
}

static void fill_layer(mmt_engine* e, LayerW& w, const std::string& p, bool decoder) {
    w.in_w = e->W(p + ".self_attn.in_proj_weight"); w.in_b = e->W(p + ".self_attn.in_proj_bias");
    w.out_w = e->W(p + ".self_attn.out_proj.weight"); w.out_b = e->W(p + ".self_attn.out_proj.bias");
    w.l1_w = e->W(p + ".linear1.weight"); w.l1_b = e->W(p + ".linear1.bias");
    w.l2_w = e->W(p + ".linear2.weight"); w.l2_b = e->W(p + ".linear2.bias");
    w.n1_w = e->W(p + ".norm1.weight"); w.n1_b = e->W(p + ".norm1.bias");
    w.n2_w = e->W(p + ".norm2.weight"); w.n2_b = e->W(p + ".norm2.bias");
    if (decoder) {
        w.ca_in_w = e->W(p + ".multihead_attn.in_proj_weight"); w.ca_in_b = e->W(p + ".multihead_attn.in_proj_bias");
        w.ca_out_w = e->W(p + ".multihead_attn.out_proj.weight"); w.ca_out_b = e->W(p + ".multihead_attn.out_proj.bias");
        w.n3_w = e->W(p + ".norm3.weight"); w.n3_b = e->W(p + ".norm3.bias");
    }
}

struct EncBuffers {
    float* X[5]; float* kb[5]; int* kidx[5]; int* nk[5];
    float* Xc; int* kidx_c; int* nk_c;
    float* ir_emb;
    float* QKV; float* ATT; float* PART; float* H;
    float* key_bias; uint8_t* pad_mask;   // chunk-local when the caller passed NULL
    // bf16 operand copies (tensor-core mode)
    __nv_bfloat16* X16[5]; __nv_bfloat16* Xc16; __nv_bfloat16* ATT16; __nv_bfloat16* H16;
};

static void plan_encoder(Arena& a, const ModeLayout& L, int Bc, int d_ff, EncBuffers& b, bool need_kb, bool need_pm, bool bf16) {
    int64_t rows_mod = 0;
    for (int m = 0; m < 5; ++m) {
        int64_t rows = L.present[m] ? (int64_t)Bc * L.S_m[m] : 0;
        b.X[m] = a.get<float>(rows * D);
        b.kb[m] = a.get<float>(rows);
        b.kidx[m] = a.get<int>(rows);
        b.nk[m] = a.get<int>(Bc);
        rows_mod += rows;
    }
    int64_t R = (int64_t)Bc * L.S_total;
    int64_t rmax = std::max(rows_mod, R);
    b.Xc = a.get<float>(R * D);
    b.kidx_c = a.get<int>(R);
    b.nk_c = a.get<int>(Bc);
    b.ir_emb = a.get<float>((int64_t)Bc * D);
    b.QKV = a.get<float>(rmax * 3 * D);
    b.key_bias = need_kb ? a.get<float>(R) : nullptr;
    b.pad_mask = need_pm ? a.get<uint8_t>(R) : nullptr;
    if (!bf16) {
        b.ATT = a.get<float>(rmax * D);
        b.PART = a.get<float>(rmax * D);
        b.H = a.get<float>(rmax * d_ff);
        for (int m = 0; m < 5; ++m) b.X16[m] = nullptr;
        b.Xc16 = b.ATT16 = b.H16 = nullptr;
    } else {
        b.ATT = b.PART = b.H = nullptr;
        for (int m = 0; m < 5; ++m) b.X16[m] = a.get<__nv_bfloat16>((L.present[m] ? (int64_t)Bc * L.S_m[m] : 0) * D);
        b.Xc16 = a.get<__nv_bfloat16>(R * D);
        b.ATT16 = a.get<__nv_bfloat16>(rmax * D);
        b.H16 = nullptr;   // the fused FFN keeps the hidden activation on the SM
    }
}

// One post-norm encoder layer over `ng` independent groups (models_MMT_v15_4.py:510-533).
struct EncGroupRun {
    float* X; int rows; int S; const float* kbias; const int* kidx; const int* nk;
    const LayerW* w; float* qkv; float* att; float* part; float* h;
    // destination of the layer output (defaults to X in place)
    float* out; int64_t stride_b, stride_s, off;
    // tensor-core mode: bf16 copies of X / attention output / FFN hidden, bf16 copy of `out`
    __nv_bfloat16 *x16, *att16, *h16, *out16;
    // ragged encoder (kernels_compact.cuh): per-sequence row ranges, key-list stride, explicit output rows
    const int *row_start, *cnt; int kstride; const int* out_rows;
    int max_keys, max_rows;   // ragged: actual per-sequence maxima (size the attention CTA: smem carve-up, threads); 0 = S
};

// Encoder self-attention launch over `ng` groups.  Shared memory and the CTA width are sized for the keys / query rows a
// sequence can actually have (ragged encoder: per-batch maxima from the index kernels) -- 60 KB instead of 151 KB per CTA
// in the cross encoder, i.e. three resident CTAs per SM instead of one for this latency-bound kernel.
static int launch_encoder_attention(mmt_engine* e, EncGroupRun* gr, int ng, int Bc, int heads, bool bf16_out, cudaStream_t s) {
    const int dh = D / heads;
    AttnParams p;
    memset(&p, 0, sizeof(p));
    p.scale = 1.0f / sqrtf((float)dh);
    int key_bound = 0, row_bound = 0;
    for (int i = 0; i < ng; ++i) {
        const bool ragged = gr[i].cnt != nullptr;
        const int kb = (ragged && gr[i].max_keys > 0) ? gr[i].max_keys : gr[i].S;
        const int rb = (ragged && gr[i].max_rows > 0) ? gr[i].max_rows : gr[i].S;
        key_bound = std::max(key_bound, kb); row_bound = std::max(row_bound, rb);
        p.g[i].qkv = gr[i].qkv; p.g[i].kbias = gr[i].kbias; p.g[i].kidx = gr[i].kidx; p.g[i].nk = gr[i].nk;
        p.g[i].out = bf16_out ? nullptr : gr[i].att; p.g[i].out16 = bf16_out ? gr[i].att16 : nullptr;
        p.g[i].S = gr[i].S;
        p.g[i].row_start = gr[i].row_start; p.g[i].cnt = gr[i].cnt; p.g[i].kstride = gr[i].kstride;
    }
    // staging capacity in keys: a 32-wide head costs 260 B per key in either kernel; sequences with more keys (MS modes with
    // every token valid: up to 902) are walked in chunks of this size
    if (dh >= 32) key_bound = std::min(key_bound, 768);
    for (int i = 0; i < ng; ++i) p.g[i].smax = key_bound;
    dim3 grid(heads, Bc, ng);
    if (dh == A5_DH && e->use_tc_attention && e->use_tc5_attention && (bf16_out || e->tc_attention_fp32)) {
        // opt-in (MMT_TC5_ATTENTION=1): tcgen05 attention, scores and output accumulators in TMEM (kernels_attn5.cuh).  Parity-tested, but
        // slower than the mma.sync kernel below at these shapes (32-wide heads, 64-key chunks: 102 vs 73 us per layer at realistic peak
        // counts, 659 vs 628 us at 582 keys, profiles/r02_attn_tc5.md): P has to round-trip through shared memory and two proxy fences
        // per chunk, and the phases of a chunk are serial within a CTA.
        MMT_TRY(tc_init(e));
        prof_pre(e, s);
        attn_encoder_tc5<<<grid, A5_THREADS, A5_SMEM_BYTES, s>>>(p);
        return check_launch(e, "attn_encoder_tc5", s);
    }
    if (dh == AT_DH && e->use_tc_attention && (bf16_out || e->tc_attention_fp32)) {   // encoder_cross in the tensor-core mode: mma.sync flash attention, two-term operand splits
        const size_t smem_tc = at_smem_bytes(key_bound);
        const int warps = std::min(12, std::max(1, (row_bound + 15) / 16));   // one 16-row tile per warp for realistic peak counts; <= 85 registers: two CTAs per SM
        MMT_CUDA(cudaFuncSetAttribute(attn_encoder_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
        MMT_CUDA(cudaFuncSetAttribute(attn_encoder_tc, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        prof_pre(e, s);
        attn_encoder_tc<<<grid, warps * 32, smem_tc, s>>>(p);
        return check_launch(e, "attn_encoder_tc", s);
    }
    if (dh == 8 && e->use_tc_attention && (bf16_out || e->tc_attention_fp32)) {   // modality encoders: same scheme on m16n8k8 tiles
        const size_t smem_tc = at8_smem_bytes(key_bound);
        const int warps = std::min(4, std::max(1, (row_bound + 15) / 16));
        MMT_CUDA(cudaFuncSetAttribute(attn_encoder_tc8, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
        prof_pre(e, s);
        attn_encoder_tc8<<<grid, warps * 32, smem_tc, s>>>(p);
        return check_launch(e, "attn_encoder_tc8", s);
    }
    const size_t smem = (size_t)key_bound * (2 * dh + 1) * sizeof(float);
    const int threads = std::min(256, std::max(64, (row_bound + 31) / 32 * 32));
    if (dh == 8) {
        MMT_CUDA(cudaFuncSetAttribute(attn_encoder_f32<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        prof_pre(e, s);
        attn_encoder_f32<8><<<grid, threads, smem, s>>>(p);
    } else if (dh == 32) {
        MMT_CUDA(cudaFuncSetAttribute(attn_encoder_f32<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        prof_pre(e, s);
        attn_encoder_f32<32><<<grid, threads, smem, s>>>(p);
    } else if (dh == 16) {
        MMT_CUDA(cudaFuncSetAttribute(attn_encoder_f32<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        prof_pre(e, s);
        attn_encoder_f32<16><<<grid, threads, smem, s>>>(p);
    } else MMT_FAIL("unsupported head dim " + std::to_string(dh));
    return check_launch(e, "attn_encoder_f32", s);
}

static int encoder_layer_fp32(mmt_engine* e, EncGroupRun* gr, int ng, int Bc, int heads, int d_ff, cudaStream_t s) {
    int maxM = 0;
    for (int i = 0; i < ng; ++i) maxM = std::max(maxM, gr[i].rows);
    {   // QKV projection
        GemmParams p = gemm_params(3 * D, D, 3 * D, 0);
        for (int i = 0; i < ng; ++i) { p.g[i].A = gr[i].X; p.g[i].lda = D; p.g[i].W = gr[i].w->in_w; p.g[i].bias = gr[i].w->in_b; p.g[i].C = gr[i].qkv; p.g[i].M = gr[i].rows; }
        MMT_TRY(launch_gemm(e, p, ng, maxM, s));
    }
    MMT_TRY(launch_encoder_attention(e, gr, ng, Bc, heads, false, s));
    {   // out-proj -> +residual -> LN1 (in place on X)
        GemmParams p = gemm_params(D, D, D, 0);
        for (int i = 0; i < ng; ++i) { p.g[i].A = gr[i].att; p.g[i].lda = D; p.g[i].W = gr[i].w->out_w; p.g[i].C = gr[i].part; p.g[i].M = gr[i].rows; }
        MMT_TRY(launch_gemm(e, p, ng, maxM, s));
        LnParams q;
        memset(&q, 0, sizeof(q));
        q.splits = 1; q.eps = 1e-5f;
        for (int i = 0; i < ng; ++i) {
            LnGroup& g = q.g[i];
            g.part = gr[i].part; g.bias = gr[i].w->out_b; g.res = gr[i].X; g.gamma = gr[i].w->n1_w; g.beta = gr[i].w->n1_b;
            g.out = gr[i].X; g.M = gr[i].rows; g.S_in = gr[i].rows > 0 ? gr[i].rows : 1; g.stride_b = 0; g.stride_s = 1; g.off = 0;
        }
        MMT_TRY(launch_ln(e, q, ng, maxM, s));
    }
    {   // FFN
        GemmParams p = gemm_params(d_ff, D, d_ff, 1);
        for (int i = 0; i < ng; ++i) { p.g[i].A = gr[i].X; p.g[i].lda = D; p.g[i].W = gr[i].w->l1_w; p.g[i].bias = gr[i].w->l1_b; p.g[i].C = gr[i].h; p.g[i].M = gr[i].rows; }
        MMT_TRY(launch_gemm(e, p, ng, maxM, s));
        GemmParams p2 = gemm_params(D, d_ff, D, 0);
        for (int i = 0; i < ng; ++i) { p2.g[i].A = gr[i].h; p2.g[i].lda = d_ff; p2.g[i].W = gr[i].w->l2_w; p2.g[i].C = gr[i].part; p2.g[i].M = gr[i].rows; }
        MMT_TRY(launch_gemm(e, p2, ng, maxM, s));
        LnParams q;
        memset(&q, 0, sizeof(q));
        q.splits = 1; q.eps = 1e-5f;
        for (int i = 0; i < ng; ++i) {
            LnGroup& g = q.g[i];
            g.part = gr[i].part; g.bias = gr[i].w->l2_b; g.res = gr[i].X; g.gamma = gr[i].w->n2_w; g.beta = gr[i].w->n2_b;
            g.out = gr[i].out ? gr[i].out : gr[i].X; g.M = gr[i].rows;
            if (gr[i].out) { g.S_in = gr[i].S; g.stride_b = gr[i].stride_b; g.stride_s = gr[i].stride_s; g.off = gr[i].off; g.out_rows = gr[i].out_rows; }
            else { g.S_in = gr[i].rows > 0 ? gr[i].rows : 1; g.stride_b = 0; g.stride_s = 1; g.off = 0; }
        }
        MMT_TRY(launch_ln(e, q, ng, maxM, s));
    }
    return 0;
}

// The same layer with every projection on the tensor cores (bf16 operands, fp32 accumulate);
// residual stream, LayerNorm statistics and the attention softmax stay fp32.
static int encoder_layer_bf16(mmt_engine* e, EncGroupRun* gr, int ng, int Bc, int heads, int d_ff, cudaStream_t s) {
    for (int i = 0; i < ng; ++i) {   // QKV projection -> fp32 (the attention kernel's softmax input)
        TcGemmParams p = tc_params(gr[i].rows, 3 * D, D);
        p.bias = gr[i].w->in_b; p.out_f32 = gr[i].qkv; p.ld_f32 = 3 * D;
        MMT_TRY(launch_tc(e, p, gr[i].x16, D, e->Wb(gr[i].w->in_w), TC_EPI_STORE, s, e->Wlo(gr[i].w->in_w)));
    }
    MMT_TRY(launch_encoder_attention(e, gr, ng, Bc, heads, true, s));
    for (int i = 0; i < ng; ++i) {   // out-proj + residual + LN1, in place on X (fp32) and X16
        TcGemmParams p = tc_params(gr[i].rows, D, D);
        p.bias = gr[i].w->out_b; p.res = gr[i].X; p.gamma = gr[i].w->n1_w; p.beta = gr[i].w->n1_b;
        p.out_f32 = gr[i].X; p.ld_f32 = D; p.out_b16 = gr[i].x16; p.ld_b16 = D;
        MMT_TRY(launch_tc(e, p, gr[i].att16, D, e->Wb(gr[i].w->out_w), TC_EPI_LN, s, e->Wlo(gr[i].w->out_w)));
    }
    for (int i = 0; i < ng; ++i) {   // fused FFN (hidden activation stays on the SM) + residual + LN2
        FfnParams p = ffn_params(gr[i].rows, d_ff);
        p.b1 = gr[i].w->l1_b; p.bias = gr[i].w->l2_b; p.res = gr[i].X; p.gamma = gr[i].w->n2_w; p.beta = gr[i].w->n2_b;
        if (gr[i].out || gr[i].out16) {
            p.out_f32 = gr[i].out; p.out_b16 = gr[i].out16;
            p.S_in = gr[i].S; p.stride_b = gr[i].stride_b; p.stride_s = gr[i].stride_s; p.off = gr[i].off; p.out_rows = gr[i].out_rows;
        } else {
            p.out_f32 = gr[i].X; p.out_b16 = gr[i].x16;
        }
        const bool one = e->enc_ffn_single;      // hi weight term only (DESIGN.md 4.3: the lo term of the FFN weights does not show in the error)
        MMT_TRY(launch_ffn(e, p, gr[i].x16, D, e->Wb(gr[i].w->l1_w), one ? nullptr : e->Wlo(gr[i].w->l1_w), e->Wb(gr[i].w->l2_w), one ? nullptr : e->Wlo(gr[i].w->l2_w), TC_EPI_LN, s));
    }
    return 0;
}

// Ragged encoder (kernels_compact.cuh): the same computation on the distinct token rows only.  Returns 0 on
// success, 1 on error, 2 when the batch does not qualify (padded rows with differing raw inputs) and the caller
// must take the dense path.
static int encode_chunk_compact(mmt_engine* e, const mmt_spectra& in, int b0, int Bc, int B_total, const ModeLayout& L,
                                float* d_memory, float* d_embedding_src, float* d_key_bias, uint8_t* d_pad_mask, bool bf16, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    const int P = d.pad_points;
    int maxS = 0;
    for (int m = 0; m < 5; ++m) maxS = std::max(maxS, L.S_m[m]);
    if (maxS > CP_SMAX) return 2;
    // ---- workspace (activation buffers sized for the dense row counts: upper bounds known without a sync)
    Arena a;
    struct { int *cnt, *nkeys, *d2c, *kidx, *flag, *row_start, *cstart, *moff, *nk_c, *ccnt, *totals, *out_rows, *kidx_c; } ix;
    float *X[5], *Xc, *ir_emb, *QKV, *ATT, *PART, *H, *key_bias_l; uint8_t* pad_mask_l;
    __nv_bfloat16 *X16[5], *Xc16, *ATT16;
    const int64_t R = (int64_t)Bc * L.S_total;
    auto plan = [&]() {
        ix.cnt = a.get<int>(5 * Bc); ix.nkeys = a.get<int>(5 * Bc);
        ix.d2c = a.get<int>((size_t)5 * Bc * CP_SMAX); ix.kidx = a.get<int>((size_t)5 * Bc * CP_SMAX);
        ix.flag = a.get<int>(1); ix.row_start = a.get<int>(5 * (Bc + 1)); ix.cstart = a.get<int>(Bc + 1);
        ix.moff = a.get<int>(5 * Bc); ix.nk_c = a.get<int>(Bc); ix.ccnt = a.get<int>(Bc); ix.totals = a.get<int>(16);
        ix.out_rows = a.get<int>((size_t)5 * Bc * maxS); ix.kidx_c = a.get<int>(R);
        int64_t rows_mod = 0;
        for (int m = 0; m < 5; ++m) { X[m] = a.get<float>((size_t)Bc * L.S_m[m] * D); rows_mod += (int64_t)Bc * L.S_m[m]; }
        const int64_t rmax = std::max(rows_mod, R);
        Xc = a.get<float>(R * D);
        ir_emb = a.get<float>((size_t)Bc * D);
        QKV = a.get<float>(rmax * 3 * D);
        key_bias_l = d_key_bias ? nullptr : a.get<float>(R);
        pad_mask_l = d_pad_mask ? nullptr : a.get<uint8_t>(R);
        if (bf16) {
            ATT = PART = H = nullptr;
            for (int m = 0; m < 5; ++m) X16[m] = a.get<__nv_bfloat16>((size_t)Bc * L.S_m[m] * D);
            Xc16 = a.get<__nv_bfloat16>(R * D);
            ATT16 = a.get<__nv_bfloat16>(rmax * D);
        } else {
            ATT = a.get<float>(rmax * D); PART = a.get<float>(rmax * D); H = a.get<float>(rmax * d.d_ff);
            for (int m = 0; m < 5; ++m) X16[m] = nullptr;
            Xc16 = ATT16 = nullptr;
        }
    };
    MMT_TRY(plan_arena(e, a, plan));
    float* key_bias = d_key_bias ? d_key_bias + (int64_t)b0 * L.S_total : key_bias_l;
    uint8_t* pad_mask = d_pad_mask ? d_pad_mask + (int64_t)b0 * L.S_total : pad_mask_l;

    const float* srcs[4] = {in.d_src_1H, in.d_src_13C, in.d_src_HSQC, in.d_src_COSY};
    const float* masks[4] = {in.d_mask_1H, in.d_mask_13C, in.d_mask_HSQC, in.d_mask_COSY};
    for (int m = 0; m < 4; ++m) if (!srcs[m] || !masks[m]) MMT_FAIL("spectra pointer missing for a modality in training_mode");
    if (!in.d_src_IR) MMT_FAIL("src_IR missing");
    if (L.has_MF && (!in.d_src_MF || !in.d_mask_MF)) MMT_FAIL("src_MF / mask_MF missing");
    if (L.has_MS && (!in.d_src_MS || !in.d_mask_MS)) MMT_FAIL("src_MS / mask_MS missing");
    if (L.has_MW && !in.d_trg_MW) MMT_FAIL("trg_MW missing");

    // ---- index maps, then one small device-to-host read of the row totals
    {
        MMT_CUDA(cudaMemsetAsync(ix.flag, 0, sizeof(int), s));
        CompactParams p;
        memset(&p, 0, sizeof(p));
        for (int m = 0; m < 4; ++m) {
            const int cols = (m == 1) ? 1 : 2;
            p.mask[m] = masks[m] + (int64_t)b0 * P; p.src[m] = srcs[m] + (int64_t)b0 * P * cols; p.cols[m] = cols;
        }
        if (L.has_MF) { p.mask_MF = in.d_mask_MF + (int64_t)b0 * P; p.src_MF = in.d_src_MF + (int64_t)b0 * P; }
        if (L.has_MS) { p.mask_MS = in.d_mask_MS + (int64_t)b0 * P; p.src_MS = in.d_src_MS + (int64_t)b0 * P; }
        for (int m = 0; m < 5; ++m) { p.present[m] = 1; p.n_x[m] = L.n_x[m]; }
        p.has_MF = L.has_MF; p.has_MS = L.has_MS; p.has_MW = L.has_MW; p.P = P; p.B = Bc;
        p.cnt = ix.cnt; p.nkeys = ix.nkeys; p.d2c = ix.d2c; p.kidx = ix.kidx; p.flag = ix.flag;
        prof_pre(e, s);
        compact_index<<<dim3(Bc, 5), 32, 0, s>>>(p);
        MMT_TRY(check_launch(e, "compact_index", s));
        CompactScanParams q;
        q.cnt = ix.cnt; q.nkeys = ix.nkeys; q.B = Bc; q.row_start = ix.row_start; q.cstart = ix.cstart; q.moff = ix.moff;
        q.nk_c = ix.nk_c; q.ccnt = ix.ccnt; q.totals = ix.totals; q.flag = ix.flag;
        prof_pre(e, s);
        compact_scan<<<1, 256, 0, s>>>(q);
        MMT_TRY(check_launch(e, "compact_scan", s));
        CompactCrossParams c;
        c.cnt = ix.cnt; c.nkeys = ix.nkeys; c.kidx = ix.kidx; c.row_start = ix.row_start; c.cstart = ix.cstart; c.moff = ix.moff; c.B = Bc;
        c.out_rows = ix.out_rows; c.out_rows_stride = (int64_t)Bc * maxS; c.kidx_c = ix.kidx_c; c.kc_stride = L.S_total;
        prof_pre(e, s);
        compact_cross_index<<<Bc, 32, 0, s>>>(c);
        MMT_TRY(check_launch(e, "compact_cross_index", s));
        MMT_CUDA(cudaMemcpyAsync(e->h_pinned, ix.totals, 16 * sizeof(int), cudaMemcpyDeviceToHost, s));
        MMT_CUDA(cudaStreamSynchronize(s));
    }
    int rows_m[5];
    for (int m = 0; m < 5; ++m) rows_m[m] = e->h_pinned[m];
    const int rows_c = e->h_pinned[5];
    if (e->h_pinned[6] != 0) return 2;
    const int max_keys_c = e->h_pinned[7], max_rows_c = e->h_pinned[8];
    int max_rows_m = 0;
    for (int m = 0; m < 5; ++m) max_rows_m = std::max(max_rows_m, e->h_pinned[9 + m]);

    // ---- IR projection 1000 -> 128 (+ReLU)
    {
        GemmParams p = gemm_params(D, d.ir_bins, D, 1);
        p.g[0].A = in.d_src_IR + (int64_t)b0 * d.ir_bins; p.g[0].lda = d.ir_bins;
        p.g[0].W = e->W(std::string(kEmbedKeys[4]) + ".weight"); p.g[0].bias = e->W(std::string(kEmbedKeys[4]) + ".bias");
        p.g[0].C = ir_emb; p.g[0].M = Bc;
        MMT_TRY(launch_gemm(e, p, 1, Bc, s));
    }
    {   // embed: dense key bias / pad mask / embedding_src outputs, compact X rows
        EmbedParams p;
        memset(&p, 0, sizeof(p));
        const float* esrc[5] = {srcs[0], srcs[1], srcs[2], srcs[3], ir_emb};
        for (int m = 0; m < 5; ++m) {
            EmbedGroup& g = p.g[m];
            g.present = 1; g.kind = (m == 4) ? 2 : (m == 1 ? 1 : 0);
            g.S_m = L.S_m[m]; g.n_x = L.n_x[m]; g.off = L.off[m]; g.blank_is_ir = (m == 4);
            if (m < 4) {
                const int cols = (m == 1) ? 1 : 2;
                g.src = esrc[m] + (int64_t)b0 * P * cols; g.mask = masks[m] + (int64_t)b0 * P;
                g.W = e->W(std::string(kEmbedKeys[m]) + ".weight"); g.b = e->W(std::string(kEmbedKeys[m]) + ".bias");
            } else {
                g.src = ir_emb;
            }
            g.X = X[m]; g.kbias = nullptr;
            g.d2c = ix.d2c + (size_t)m * Bc * CP_SMAX; g.row_start = ix.row_start + m * (Bc + 1);
        }
        p.has_MF = L.has_MF; p.has_MS = L.has_MS; p.has_MW = L.has_MW;
        if (L.has_MF) { p.src_MF = in.d_src_MF + (int64_t)b0 * P; p.mask_MF = in.d_mask_MF + (int64_t)b0 * P; p.E_MF = e->W("linear_embedding_MF.embedding.weight"); p.mf_vocab = d.mf_vocab; }
        if (L.has_MS) { p.src_MS = in.d_src_MS + (int64_t)b0 * P; p.mask_MS = in.d_mask_MS + (int64_t)b0 * P; p.E_MS = e->W("linear_embedding_MS.embedding.weight"); p.ms_vocab = d.ms_vocab; }
        if (L.has_MW) {
            p.trg_MW = in.d_trg_MW + b0;
            p.W_MW = e->W("linear_embedding_MW.linear_spec_embedding_MW.weight");
            p.b_MW = e->W("linear_embedding_MW.linear_spec_embedding_MW.bias");
        }
        p.B = Bc; p.S_total = L.S_total; p.P = P; p.float_mask = 0;
        p.cross_X = Xc; p.key_bias = key_bias; p.pad_mask = pad_mask;
        p.embedding_src = d_embedding_src; p.B_total = B_total; p.b0 = b0;
        prof_pre(e, s);
        embed_tokens<<<dim3(Bc, 5), 128, 0, s>>>(p);
        MMT_TRY(check_launch(e, "embed_tokens", s));
    }
    if (bf16)
        for (int m = 0; m < 5; ++m) {
            prof_pre(e, s);
            pack_rows_bf16<<<(unsigned)((rows_m[m] + 7) / 8), 256, 0, s>>>(X[m], nullptr, D, rows_m[m], X16[m]);
            MMT_TRY(check_launch(e, "pack_rows_bf16", s));
        }
    // ---- five modality encoders on their compact rows
    {
        EncGroupRun gr[5];
        int64_t row_off = 0;
        for (int m = 0; m < 5; ++m) {
            EncGroupRun& g = gr[m];
            memset(&g, 0, sizeof(g));
            g.X = X[m]; g.rows = rows_m[m]; g.S = L.S_m[m];
            g.kbias = nullptr; g.kidx = ix.kidx + (size_t)m * Bc * CP_SMAX; g.nk = ix.nkeys + m * Bc;
            g.row_start = ix.row_start + m * (Bc + 1); g.cnt = ix.cnt + m * Bc; g.kstride = CP_SMAX;
            g.max_keys = max_rows_m; g.max_rows = max_rows_m;
            g.qkv = QKV + row_off * 3 * D;
            if (bf16) { g.x16 = X16[m]; g.att16 = ATT16 + row_off * D; }
            else { g.att = ATT + row_off * D; g.part = PART + row_off * D; g.h = H + row_off * d.d_ff; }
            row_off += g.rows;
        }
        auto set_layer = [&](int m, int l) {
            gr[m].w = &e->enc[m][l];
            if (l == d.n_enc_layers - 1) {   // last layer scatters into the spectrum-major cross buffer
                gr[m].out = Xc; gr[m].out16 = Xc16; gr[m].out_rows = ix.out_rows + (size_t)m * Bc * maxS;
                gr[m].stride_b = 0; gr[m].stride_s = 1; gr[m].off = 0;
            }
        };
        if (e->use_enc_streams && !e->profiling) {
            // The five stacks are independent until encoder_cross and each is a chain of small launches (30-100 row
            // tiles on 148 SMs): run them as five concurrent chains on forked streams, joined before the cross encoder.
            for (int m = 0; m < 5; ++m) if (!e->enc_stream[m]) MMT_CUDA(cudaStreamCreateWithFlags(&e->enc_stream[m], cudaStreamNonBlocking));
            for (int m = 0; m < 6; ++m) if (!e->enc_ev[m]) MMT_CUDA(cudaEventCreateWithFlags(&e->enc_ev[m], cudaEventDisableTiming));
            MMT_CUDA(cudaEventRecord(e->enc_ev[5], s));
            for (int m = 0; m < 5; ++m) {
                cudaStream_t sm = e->enc_stream[m];
                MMT_CUDA(cudaStreamWaitEvent(sm, e->enc_ev[5], 0));
                gr[m].max_keys = gr[m].max_rows = e->h_pinned[9 + m];      // this stack's own maxima size its attention CTAs
                for (int l = 0; l < d.n_enc_layers; ++l) {
                    set_layer(m, l);
                    if (bf16) MMT_TRY(encoder_layer_bf16(e, &gr[m], 1, Bc, d.n_heads, d.d_ff, sm));
                    else MMT_TRY(encoder_layer_fp32(e, &gr[m], 1, Bc, d.n_heads, d.d_ff, sm));
                }
                MMT_CUDA(cudaEventRecord(e->enc_ev[m], sm));
            }
            for (int m = 0; m < 5; ++m) MMT_CUDA(cudaStreamWaitEvent(s, e->enc_ev[m], 0));
        } else {
            for (int l = 0; l < d.n_enc_layers; ++l) {
                for (int m = 0; m < 5; ++m) set_layer(m, l);
                if (bf16) MMT_TRY(encoder_layer_bf16(e, gr, 5, Bc, d.n_heads, d.d_ff, s));
                else MMT_TRY(encoder_layer_fp32(e, gr, 5, Bc, d.n_heads, d.d_ff, s));
            }
        }
    }
    // ---- encoder_cross on the concatenated compact rows
    {
        EncGroupRun g;
        memset(&g, 0, sizeof(g));
        g.X = Xc; g.rows = rows_c; g.S = L.S_total; g.kbias = nullptr; g.kidx = ix.kidx_c; g.nk = ix.nk_c;
        g.row_start = ix.cstart; g.cnt = ix.ccnt; g.kstride = L.S_total;
        g.max_keys = max_keys_c; g.max_rows = max_rows_c;
        g.qkv = QKV; g.att = ATT; g.part = PART; g.h = H;
        g.x16 = Xc16; g.att16 = ATT16;
        for (int l = 0; l < d.n_enc_layers; ++l) {
            g.w = &e->enc[5][l];
            if (bf16) MMT_TRY(encoder_layer_bf16(e, &g, 1, Bc, d.n_heads_cross, d.d_ff, s));
            else MMT_TRY(encoder_layer_fp32(e, &g, 1, Bc, d.n_heads_cross, d.d_ff, s));
        }
    }
    {   // replicate the padded rows while writing the sequence-first (S, B, 128) memory
        ExpandParams p;
        memset(&p, 0, sizeof(p));
        p.Y = Xc; p.cstart = ix.cstart; p.moff = ix.moff; p.d2c = ix.d2c; p.B = Bc; p.S_total = L.S_total;
        for (int m = 0; m < 5; ++m) { p.off[m] = L.off[m]; p.S_m[m] = L.S_m[m]; }
        p.memory = d_memory; p.B_total = B_total; p.b0 = b0;
        prof_pre(e, s);
        expand_memory<<<(unsigned)((R + 7) / 8), 256, 0, s>>>(p);
        MMT_TRY(check_launch(e, "expand_memory", s));
    }
    return 0;
}

static int encode_chunk(mmt_engine* e, const mmt_spectra& in, int b0, int Bc, int B_total, uint32_t mode, const ModeLayout& L,
                        float* d_memory, float* d_embedding_src, float* d_key_bias, uint8_t* d_pad_mask, bool bf16, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    const int P = d.pad_points;
    Arena a;
    EncBuffers b;
    MMT_TRY(plan_arena(e, a, [&]() { plan_encoder(a, L, Bc, d.d_ff, b, d_key_bias == nullptr, d_pad_mask == nullptr, bf16); }));
    float* key_bias = d_key_bias ? d_key_bias + (int64_t)b0 * L.S_total : b.key_bias;
    uint8_t* pad_mask = d_pad_mask ? d_pad_mask + (int64_t)b0 * L.S_total : b.pad_mask;

    // IR projection 1000 -> 128 (+ReLU)   (models_MMT_v15_4.py:437-444, 761-767)
    if (L.present[4]) {
        GemmParams p = gemm_params(D, d.ir_bins, D, 1);
        p.g[0].A = in.d_src_IR + (int64_t)b0 * d.ir_bins; p.g[0].lda = d.ir_bins;
        p.g[0].W = e->W(std::string(kEmbedKeys[4]) + ".weight"); p.g[0].bias = e->W(std::string(kEmbedKeys[4]) + ".bias");
        p.g[0].C = b.ir_emb; p.g[0].M = Bc;
        MMT_TRY(launch_gemm(e, p, 1, Bc, s));
    }
    {   // embed + concatenate
        EmbedParams p;
        memset(&p, 0, sizeof(p));
        const float* srcs[5] = {in.d_src_1H, in.d_src_13C, in.d_src_HSQC, in.d_src_COSY, b.ir_emb};
        const float* masks[5] = {in.d_mask_1H, in.d_mask_13C, in.d_mask_HSQC, in.d_mask_COSY, nullptr};
        for (int m = 0; m < 5; ++m) {
            EmbedGroup& g = p.g[m];
            g.present = L.present[m]; g.kind = (m == 4) ? 2 : (m == 1 ? 1 : 0);
            g.S_m = L.S_m[m]; g.n_x = L.n_x[m]; g.off = L.off[m]; g.blank_is_ir = (m == 4);
            if (!g.present) continue;
            if (m < 4) {
                if (!srcs[m] || !masks[m]) MMT_FAIL("spectra pointer missing for a modality in training_mode");
                int cols = (m == 1) ? 1 : 2;
                g.src = srcs[m] + (int64_t)b0 * P * cols; g.mask = masks[m] + (int64_t)b0 * P;
                g.W = e->W(std::string(kEmbedKeys[m]) + ".weight"); g.b = e->W(std::string(kEmbedKeys[m]) + ".bias");
            } else {
                g.src = b.ir_emb;
            }
            g.X = b.X[m]; g.kbias = b.kb[m];
        }
        p.has_MF = L.has_MF; p.has_MS = L.has_MS; p.has_MW = L.has_MW;
        if (L.has_MF) {
            if (!in.d_src_MF || !in.d_mask_MF) MMT_FAIL("src_MF / mask_MF missing");
            p.src_MF = in.d_src_MF + (int64_t)b0 * P; p.mask_MF = in.d_mask_MF + (int64_t)b0 * P;
            p.E_MF = e->W("linear_embedding_MF.embedding.weight"); p.mf_vocab = d.mf_vocab;
        }
        if (L.has_MS) {
            if (!in.d_src_MS || !in.d_mask_MS) MMT_FAIL("src_MS / mask_MS missing");
            p.src_MS = in.d_src_MS + (int64_t)b0 * P; p.mask_MS = in.d_mask_MS + (int64_t)b0 * P;
            p.E_MS = e->W("linear_embedding_MS.embedding.weight"); p.ms_vocab = d.ms_vocab;
        }
        if (L.has_MW) {
            if (!in.d_trg_MW) MMT_FAIL("trg_MW missing");
            p.trg_MW = in.d_trg_MW + b0;
            p.W_MW = e->W("linear_embedding_MW.linear_spec_embedding_MW.weight");
            p.b_MW = e->W("linear_embedding_MW.linear_spec_embedding_MW.bias");
        }
        p.B = Bc; p.S_total = L.S_total; p.P = P; p.float_mask = L.float_mask;
        p.cross_X = b.Xc; p.key_bias = key_bias; p.pad_mask = pad_mask;
        p.embedding_src = d_embedding_src; p.B_total = B_total; p.b0 = b0;
        prof_pre(e, s);
        embed_tokens<<<dim3(Bc, 5), 128, 0, s>>>(p);
        MMT_TRY(check_launch(e, "embed_tokens", s));
    }
    if (!d_memory) return 0;   // embedding-only call (forward()'s 2nd output for an encode served from the cache)
    {   // key compaction for the modality encoders and encoder_cross
        KeyIndexParams p;
        memset(&p, 0, sizeof(p));
        int ng = 0;
        for (int m = 0; m < 5; ++m) if (L.present[m]) { p.g[ng].kbias = b.kb[m]; p.g[ng].kidx = b.kidx[m]; p.g[ng].nk = b.nk[m]; p.g[ng].S = L.S_m[m]; ++ng; }
        p.g[ng].kbias = key_bias; p.g[ng].kidx = b.kidx_c; p.g[ng].nk = b.nk_c; p.g[ng].S = L.S_total; ++ng;
        p.B = Bc;
        prof_pre(e, s);
        build_key_index<<<dim3(Bc, ng), 32, 0, s>>>(p);
        MMT_TRY(check_launch(e, "build_key_index", s));
    }
    if (bf16) {   // bf16 operand copies of the embedded tokens; blank-modality rows of the concatenated memory are zero
        bool any_blank = false;
        for (int m = 0; m < 5; ++m) {
            if (!L.present[m]) { any_blank = true; continue; }
            const int64_t rows = (int64_t)Bc * L.S_m[m];
            prof_pre(e, s);
            pack_rows_bf16<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(b.X[m], nullptr, D, rows, b.X16[m]);
            MMT_TRY(check_launch(e, "pack_rows_bf16", s));
        }
        if (any_blank) MMT_CUDA(cudaMemsetAsync(b.Xc16, 0, (size_t)Bc * L.S_total * D * sizeof(__nv_bfloat16), s));
    }
    // five modality encoders, batched as groups of one launch
    {
        EncGroupRun gr[5];
        int ng = 0;
        int64_t row_off = 0;
        for (int m = 0; m < 5; ++m) {
            if (!L.present[m]) continue;
            EncGroupRun& g = gr[ng];
            memset(&g, 0, sizeof(g));
            g.X = b.X[m]; g.rows = Bc * L.S_m[m]; g.S = L.S_m[m]; g.kbias = b.kb[m]; g.kidx = b.kidx[m]; g.nk = b.nk[m];
            g.qkv = b.QKV + row_off * 3 * D;
            if (bf16) { g.x16 = b.X16[m]; g.att16 = b.ATT16 + row_off * D; g.h16 = b.H16 + row_off * d.d_ff; }
            else { g.att = b.ATT + row_off * D; g.part = b.PART + row_off * D; g.h = b.H + row_off * d.d_ff; }
            row_off += g.rows;
            ++ng;
        }
        for (int l = 0; l < d.n_enc_layers && ng > 0; ++l) {
            int gi = 0;
            for (int m = 0; m < 5; ++m) {
                if (!L.present[m]) continue;
                gr[gi].w = &e->enc[m][l];
                if (l == d.n_enc_layers - 1) {   // last layer writes into the concatenated memory [Bc][S_total][D]
                    gr[gi].out = b.Xc; gr[gi].out16 = b.Xc16; gr[gi].stride_b = L.S_total; gr[gi].stride_s = 1; gr[gi].off = L.off[m];
                }
                ++gi;
            }
            if (bf16) MMT_TRY(encoder_layer_bf16(e, gr, ng, Bc, d.n_heads, d.d_ff, s));
            else MMT_TRY(encoder_layer_fp32(e, gr, ng, Bc, d.n_heads, d.d_ff, s));
        }
    }
    // encoder_cross over the concatenated memory (models_MMT_v15_4.py:941-944)
    {
        EncGroupRun g;
        memset(&g, 0, sizeof(g));
        g.X = b.Xc; g.rows = Bc * L.S_total; g.S = L.S_total; g.kbias = key_bias; g.kidx = b.kidx_c; g.nk = b.nk_c;
        g.qkv = b.QKV; g.att = b.ATT; g.part = b.PART; g.h = b.H;
        g.x16 = b.Xc16; g.att16 = b.ATT16; g.h16 = b.H16;
        for (int l = 0; l < d.n_enc_layers; ++l) {
            g.w = &e->enc[5][l];
            if (l == d.n_enc_layers - 1) { g.out = d_memory; g.out16 = nullptr; g.stride_b = 1; g.stride_s = B_total; g.off = b0; }   // (S,B,D)
            if (bf16) MMT_TRY(encoder_layer_bf16(e, &g, 1, Bc, d.n_heads_cross, d.d_ff, s));
            else MMT_TRY(encoder_layer_fp32(e, &g, 1, Bc, d.n_heads_cross, d.d_ff, s));
        }
    }
    return 0;
}

// ---------------------------------------------------------------------------
// decoder
// ---------------------------------------------------------------------------
struct DecBuffers {
    float *x, *qkv, *att, *part, *qc, *h;
    int64_t part_rows;                 // capacity of `part` in rows of D floats
    char* kv_pool; int* block_table;   // paged self-attention cache, a pool of kv_esz-byte elements per layer (layer_pool)
    int64_t pool_pages;                // pages per layer pool (Nw * pps; twice that for the beam search's copy-on-write parity)
    int kv_first;                      // first layer with a pool: 1 when every wave of the run takes layer 0 from the table
    uint8_t* hist; int hist_ld;        // layer 0 on the position x token table: token history [col][hist_ld] (nullptr otherwise)
    char* cross_kv;                    // projected memory [layer][K|V][head][row][dh], kv_esz-byte elements
    size_t kv_esz;                     // 4 (fp32 check mode) | 2 (bf16 tensor-core mode)
    int *nk, *row_start; int64_t* row_off; float* kbias_c;
    int* ctl;   // [0] step, [1] done_ctas, [8..8+max_len) nonpad counts
    uint64_t* rng_state;   // {philox seed, offset of step 0} of this call (read by the sampler from device memory)
    // bf16 operand copies (tensor-core mode)
    __nv_bfloat16 *x16, *att16, *h16, *mem16;
    // stop at <EOS> (mmt_decode_until_eos, kernels_retire.cuh), nullptr / 0 otherwise.  plan_rows: the wave's starting size,
    // which fixes every kernel-variant decision of the un-fused step through its compactions (bit identity with the plain
    // call).  orig / col_start / col_count: the compacted wave's row -> sequence map and per-column rows (nullptr until the
    // first compaction).  eos_len: first-<EOS> step per sequence of the lane.  rt_*: compaction storage.
    int64_t plan_rows;
    const int *orig, *col_start, *col_count;
    int* eos_len;
    int *rt_orig[2], *rt_bt, *rt_src, *rt_col_start, *rt_col_count;
};
constexpr int MAX_SPLITS = 32;

// l0_table: the run's un-fused waves take layer 0 from the table (token history); l0_pool: a wave may need layer 0's pages
static void plan_decoder(Arena& a, const mmt_model_desc& d, int64_t Nw, int Bmw, int S, int max_len, DecBuffers& b, bool bf16, int fused_rows, int kv_copies = 1,
                         bool retire = false, bool l0_table = false, bool l0_pool = true) {
    const int L = d.n_dec_layers;
    const int pps = (max_len + PAGE_TOKENS - 1) / PAGE_TOKENS;
    b.x = a.get<float>(Nw * D);
    b.qkv = a.get<float>(Nw * 3 * D);
    b.att = a.get<float>(Nw * D);
    // FFN2 split partials exist for small waves only (fused step: Nw <= fused_rows; un-fused step: M < 2048) -- but a run
    // planned for a large wave can end in a short one (17,408 sequences = 16,384 + 1,024), so the buffer is sized for the
    // largest small wave this plan can meet, not for the planned wave alone
    b.part_rows = std::max<int64_t>(Nw, std::min<int64_t>(Nw, std::max(fused_rows, 2048)) * MAX_SPLITS);
    b.part = a.get<float>(b.part_rows * D);
    b.qc = a.get<float>(Nw * D);
    b.h = a.get<float>(bf16 ? 0 : Nw * d.d_ff);
    b.kv_esz = bf16 ? 2 : 4;
    b.pool_pages = (int64_t)kv_copies * Nw * pps;
    b.kv_first = l0_pool ? 0 : 1;
    b.kv_pool = a.get<char>((size_t)(L - b.kv_first) * b.pool_pages * 2 * PAGE_TOKENS * D * b.kv_esz);
    b.hist_ld = pps * PAGE_TOKENS;
    b.hist = l0_table ? a.get<uint8_t>((size_t)Nw * b.hist_ld) : nullptr;
    b.block_table = a.get<int>(Nw * pps);
    int64_t R = (int64_t)Bmw * S;
    b.cross_kv = a.get<char>((size_t)L * 2 * R * D * b.kv_esz);
    b.nk = a.get<int>(Bmw);
    b.row_start = a.get<int>(Bmw);
    b.row_off = a.get<int64_t>(R);
    b.kbias_c = a.get<float>(R);
    b.ctl = a.get<int>(8 + 256);
    b.rng_state = a.get<uint64_t>(2);
    b.x16 = b.att16 = b.h16 = b.mem16 = nullptr;
    if (bf16) {
        b.x16 = a.get<__nv_bfloat16>(Nw * D);
        b.att16 = a.get<__nv_bfloat16>(Nw * D);
        b.h16 = nullptr;   // fused FFN: no hidden activation in HBM
        b.mem16 = a.get<__nv_bfloat16>(R * D);
    }
    b.plan_rows = 0; b.orig = b.col_start = b.col_count = nullptr; b.eos_len = nullptr;
    b.rt_orig[0] = b.rt_orig[1] = b.rt_bt = b.rt_src = b.rt_col_start = b.rt_col_count = nullptr;
    if (retire) {
        b.rt_orig[0] = a.get<int>(Nw); b.rt_orig[1] = a.get<int>(Nw); b.rt_bt = a.get<int>(Nw * pps); b.rt_src = a.get<int>(Nw);
        b.rt_col_start = a.get<int>(Bmw); b.rt_col_count = a.get<int>(Bmw);
    }
}

// layer l's cache pages (nullptr: layer 0 of a run that takes it from the table throughout)
static char* layer_pool(const DecBuffers& b, int l) {
    return l < b.kv_first ? nullptr : b.kv_pool + (size_t)(l - b.kv_first) * b.pool_pages * 2 * PAGE_TOKENS * D * b.kv_esz;
}

// Page map of a wave: page j of sequence n is physical page j * Nw + n ("slot-major").  At position t every sequence reads its
// pages 0 .. t / 16, so the pages a step touches form ONE contiguous region of the pool that grows with t.  With the
// sequence-major map (n * pps + j) a step read 8 KB pages at a 64 KB stride with a t-dependent duty cycle, which the HBM
// channel hash spread unevenly (ncu, t = 41: busiest channel 67 % active, idlest 33 %, profiles/r02_ncu_summary.md).
__global__ void init_block_table(int* bt, int64_t Nw, int pps) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < Nw * pps) bt[i] = (int)((i % pps) * Nw + i / pps);
}

struct DecodeRun {
    const mmt_decode_args* a;
    int mode;                 // pick: 0 greedy, 1 multinomial, 2 none (logits only)
    const int64_t* trg;       // forced input tokens (T, N_total): teacher forcing; nullptr = feed the picks back
    const int64_t* target = nullptr; float* target_prob = nullptr;   // optional (T, N_total): probability of a given token at every position
    int T;                    // steps to run
    int64_t* tokens; float* probs; float* logits;   // outputs, leading dimension N_total
    int64_t ldn = -1;         // >= 0 overrides the leading dimension (0: single-row token / logit buffers, beam search)
    bool serial_first = false;   // the step's first kernel waits for full completion of its predecessor (its prologue reads the block table)
    bool per_memory_rng = false; // multinomial draws in per-memory streams (torch_rng_row): one (n_cand, V) call per column and step
    int64_t eos = -1;            // >= 0: stop at this id (mmt_decode_until_eos): finished sequences retire from large waves
    int32_t* len = nullptr;      //   out (N) first-<EOS> positions
    int64_t* h_rows = nullptr;   //   out (T), optional: rows computed per position
    // per-column sampling controls (mmt_decode_controlled), multinomial only: validated host arrays (Bm) that run_decode
    // copies to the device arrays the sampler reads (the values stay out of the captured graph); nullptr otherwise
    const float* h_temp = nullptr; const int32_t* h_topk = nullptr; const float* h_topp = nullptr;
    const float* ctl_temp = nullptr; const int32_t* ctl_topk = nullptr; const float* ctl_topp = nullptr;
};

// Projects the memory of one wave to per-layer cross-attention K/V (head-major) once;
// the reference redoes this projection on every step (validate_generate_MMT_v15_4.py:751).
static int decode_prepare_wave(mmt_engine* e, const mmt_decode_args& a, int b0, int Bmw, DecBuffers& b, bool bf16, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    MemIndexParams mp;
    mp.key_bias = a.d_key_bias + (int64_t)b0 * a.S; mp.S = a.S; mp.Bm = Bmw;
    mp.stride_s = a.stride_s; mp.stride_b = a.stride_b;
    mp.nk = b.nk; mp.row_start = b.row_start; mp.row_off = b.row_off; mp.kbias_c = b.kbias_c;
    prof_pre(e, s);
    build_memory_index<<<Bmw, 32, 0, s>>>(mp);
    MMT_TRY(check_launch(e, "build_memory_index", s));
    const int64_t R = (int64_t)Bmw * a.S;
    const int dh = D / d.n_heads;
    if (bf16) {   // gather the un-masked memory rows into a dense bf16 operand, then one tcgen05 GEMM per layer
        prof_pre(e, s);
        pack_rows_bf16<<<(unsigned)((R + 7) / 8), 256, 0, s>>>(a.d_memory + (int64_t)b0 * a.stride_b, b.row_off, 0, R, b.mem16);
        MMT_TRY(check_launch(e, "pack_rows_bf16", s));
        for (int l = 0; l < d.n_dec_layers; ++l) {
            TcGemmParams p = tc_params((int)R, 2 * D, D);
            p.bias = e->dec[l].ca_in_b + D;
            p.out_b16 = reinterpret_cast<__nv_bfloat16*>(b.cross_kv + (size_t)l * 2 * R * D * b.kv_esz);
            p.head_major = 1; p.hm_heads = d.n_heads; p.hm_dh = dh; p.hm_rows = a.S;
            MMT_TRY(launch_tc(e, p, b.mem16, D, e->Wb(e->dec[l].ca_in_w + (int64_t)D * D), TC_EPI_STORE, s, e->Wlo(e->dec[l].ca_in_w + (int64_t)D * D)));
        }
        return 0;
    }
    for (int l = 0; l < d.n_dec_layers; ++l) {
        GemmParams p = gemm_params(2 * D, D, 0, 0);
        p.g[0].A = a.d_memory + (int64_t)b0 * a.stride_b; p.g[0].a_row_off = b.row_off; p.g[0].lda = 0;
        p.g[0].W = e->dec[l].ca_in_w + (int64_t)D * D;     // rows D..3D of in_proj: K then V
        p.g[0].bias = e->dec[l].ca_in_b + D;
        p.g[0].C = reinterpret_cast<float*>(b.cross_kv + (size_t)l * 2 * R * D * b.kv_esz); p.g[0].M = (int)R;
        p.out_mode = GEMM_OUT_HEADMAJOR; p.hm_heads = d.n_heads; p.hm_dh = dh; p.hm_rows = a.S;
        MMT_TRY(launch_gemm(e, p, 1, (int)R, s));
    }
    return 0;
}

// Decoder layer 0's input at position t is E_tok[tok] + E_pos[t]: its Q and K | V rows depend on the pair (t, tok) alone.
// The table holds them for every pair (128 x 43 = 5,504 rows: Q 2.8 MB fp32, K | V 2.8 MB bf16, small enough to stay in
// L2), made by the step's own layer-0 projection -- the same bf16 input rows, tcgen05 GEMM call, bias add and bf16
// rounding -- so that the large-wave step reads layer 0 from it bit for bit instead of projecting, appending and re-reading
// 67 MB of cache per position.  Built once, outside any capture (a fixed allocation: cached step graphs stay valid).
static int ensure_l0_table(mmt_engine* e, cudaStream_t s) {
    if (e->l0_qtab) return 0;
    cudaStreamCaptureStatus cs;
    MMT_CUDA(cudaStreamIsCapturing(s, &cs));
    if (cs != cudaStreamCaptureStatusNone) MMT_FAIL("decode: the layer-0 table is built by the first large bf16 decode, which cannot run under stream capture");
    const mmt_model_desc& d = e->desc;
    const LayerW& w = e->dec[0];
    const int64_t rows = (int64_t)d.max_len * d.vocab;
    __nv_bfloat16* x16 = nullptr;
    float* qkv = nullptr;
    float* qtab = nullptr;
    __nv_bfloat16* kvtab = nullptr;
    auto release = [&]() { cudaFree(x16); cudaFree(qkv); cudaFree(qtab); cudaFree(kvtab); };
    if (cudaMalloc(&x16, rows * D * sizeof(__nv_bfloat16)) != cudaSuccess || cudaMalloc(&qkv, rows * 3 * D * sizeof(float)) != cudaSuccess ||
        cudaMalloc(&qtab, rows * D * sizeof(float)) != cudaSuccess || cudaMalloc(&kvtab, rows * 2 * D * sizeof(__nv_bfloat16)) != cudaSuccess) {
        release();
        MMT_FAIL("decode: cudaMalloc of the layer-0 table failed");
    }
    int rc = 0;
    prof_pre(e, s);
    l0_table_rows<<<(unsigned)((rows + 3) / 4), 128, 0, s>>>(e->W("embed_trg.weight"), e->W("pe_trg.weight"), (int)d.vocab, rows, x16);
    rc = check_launch(e, "l0_table_rows", s);
    if (!rc) {     // decode_self_attention_layer's projection, every column to fp32
        TcGemmParams p = tc_params((int)rows, 3 * D, D);
        p.bias = w.in_b; p.out_f32 = qkv; p.ld_f32 = 3 * D;
        rc = launch_tc(e, p, x16, D, e->Wb(w.in_w), TC_EPI_STORE, s, e->dec_proj_single ? nullptr : e->Wlo(w.in_w));
    }
    if (!rc) {
        prof_pre(e, s);
        l0_table_split<<<(unsigned)((rows + 3) / 4), 128, 0, s>>>(qkv, rows, qtab, kvtab);
        rc = check_launch(e, "l0_table_split", s);
    }
    cudaError_t se = cudaStreamSynchronize(s);
    cudaFree(x16); cudaFree(qkv);
    x16 = nullptr; qkv = nullptr;
    if (rc || se != cudaSuccess) {
        release();
        if (rc) return rc;
        MMT_FAIL(std::string("decode: layer-0 table build failed: ") + cudaGetErrorString(se));
    }
    e->l0_qtab = qtab; e->l0_kvtab = kvtab;
    return 0;
}

// Un-fused step, one decoder layer: the QKV projection of the new position (x16 / x at step *b.ctl) and its self-attention
// over the layer's cache `pool` -> att16 (bf16) | att (fp32).  bf16: tcgen05 projection whose epilogue appends K | V to the
// token-major (default) or head-major pages, or (MMT_NO_KV_EPILOGUE) the attention kernel appends them; fp32: SIMT GEMM.
// decode_step and the unit hook mmt_decode_self_attention both run this.
// l0_table (layer 0 of the un-fused bf16 token-major step, b.hist set): no projection and no cache; the attention reads the
// rows of the sequence's (position, token) pairs from the engine's layer-0 table (ensure_l0_table, TmTable).
static int decode_self_attention_layer(mmt_engine* e, const LayerW& w, const DecBuffers& b, char* pool, int pps, int64_t Nw, bool bf16,
                                       bool pdl_u, cudaStream_t s, bool l0_table = false) {
    const int H = e->desc.n_heads, dh = D / H;
    const float scale = 1.0f / sqrtf((float)dh);
    const int* step = b.ctl;
    const int M = (int)Nw;
    if (dh != 8) MMT_FAIL("decoder head dim must be 8");
    const unsigned tm_blocks = (unsigned)((Nw * (H / 8) + 7) / 8);      // token-major / table: a warp per (sequence, 8 heads)
    if (l0_table) {
        if (!b.hist || !e->l0_qtab) MMT_FAIL("decode: layer-0 table path without its table or token history");
        const TmTable src{e->l0_qtab, e->l0_kvtab, b.hist, b.hist_ld, (int)e->desc.vocab, b.orig};
        prof_pre(e, s);
        launch_args(decode_self_attention_tm<8, TmTable>, dim3(tm_blocks), dim3(256), 0, s, pdl_u, src, Nw, H, scale, step, b.att16);
        return check_launch(e, "decode_self_attention_l0", s);
    }
    if (bf16) {   // K | V columns of the projection land in the cache pages directly; the fp32 row keeps only Q
        TcGemmParams p = tc_params(M, 3 * D, D);
        // (with the K | V columns going to the cache, the Q columns form a dense [N][D] buffer: a 512-byte row every 512
        // bytes instead of every 1536)
        p.bias = w.in_b; p.out_f32 = b.qkv; p.ld_f32 = e->use_kv_epilogue ? D : 3 * D;
        p.kv_append = e->use_kv_epilogue ? (e->kv_tok_major && H % 8 == 0 ? 2 : 1) : 0; p.kv_pool = reinterpret_cast<__nv_bfloat16*>(pool); p.block_table = b.block_table; p.pps = pps; p.step = step; p.kv_heads = H;
        MMT_TRY(launch_tc(e, p, b.x16, D, e->Wb(w.in_w), TC_EPI_STORE, s, e->dec_proj_single ? nullptr : e->Wlo(w.in_w), pdl_u));
    } else {
        GemmParams p = gemm_params(3 * D, D, 3 * D, 0);
        p.g[0].A = b.x; p.g[0].lda = D; p.g[0].W = w.in_w; p.g[0].bias = w.in_b; p.g[0].C = b.qkv; p.g[0].M = M;
        p.splits = 1; p.part_stride = Nw * D;
        MMT_TRY(launch_gemm(e, p, 1, M, s, b.plan_rows));
    }
    prof_pre(e, s);
    const unsigned sa_blocks = (unsigned)((Nw * (H / 4) + 7) / 8);     // a warp per (sequence, 4 heads)
    if (bf16 && e->use_kv_epilogue && e->kv_tok_major && H % 8 == 0)      // token-major pages: a warp per (sequence, 8 heads)
        launch_args(decode_self_attention_tm<8, TmPaged>, dim3(tm_blocks), dim3(256), 0, s, pdl_u, TmPaged{b.qkv, reinterpret_cast<const __nv_bfloat16*>(pool), b.block_table, pps}, Nw, H, scale, step, b.att16);
    else if (bf16 && e->use_kv_epilogue) launch_args(decode_self_attention_g8<8, __nv_bfloat16, false>, dim3(sa_blocks), dim3(256), 0, s, pdl_u, (const float*)b.qkv, reinterpret_cast<__nv_bfloat16*>(pool), (const int*)b.block_table, pps, Nw, H, scale, step, (float*)nullptr, b.att16);
    else if (bf16) launch_args(decode_self_attention_g8<8, __nv_bfloat16>, dim3(sa_blocks), dim3(256), 0, s, pdl_u, (const float*)b.qkv, reinterpret_cast<__nv_bfloat16*>(pool), (const int*)b.block_table, pps, Nw, H, scale, step, (float*)nullptr, b.att16);
    else decode_self_attention_g8<8, float><<<sa_blocks, 256, 0, s>>>(b.qkv, reinterpret_cast<float*>(pool), b.block_table, pps, Nw, H, scale, step, b.att, b.att16);
    return check_launch(e, "decode_self_attention", s);
}

// Un-fused step, one decoder layer: cross attention of the queries qc over the layer's projected memory `ckv` -> att16 | att.
// Candidates of a spectrum share K/V: tensor-core tiles of 16 candidates for n_cand >= 8 in the bf16 mode (MMT_NO_TC_ATTENTION:
// the SIMT kernel).  decode_step and the unit hook mmt_decode_cross_attention both run this.
static int decode_cross_attention_layer(mmt_engine* e, const mmt_decode_args& a, const DecBuffers& b, const char* ckv, int64_t Nw, int Bmw,
                                        bool bf16, bool pdl_u, cudaStream_t s) {
    const int H = e->desc.n_heads, dh = D / H;
    const float scale = 1.0f / sqrtf((float)dh);
    if (dh != 8) MMT_FAIL("decoder head dim must be 8");
    const unsigned attn_blocks = (unsigned)((Nw * H + 7) / 8);
    prof_pre(e, s);
    if (bf16 && a.n_cand >= 8 && e->use_tc_attention)
        launch_args(decode_cross_attention_tc, dim3(H, Bmw), dim3(256), dx_smem_bytes(a.S), s, pdl_u, (const float*)b.qc, reinterpret_cast<const __nv_bfloat16*>(ckv), (int64_t)a.S, (const int*)b.nk, (const int*)b.row_start, (const float*)b.kbias_c, (int)a.n_cand, H, scale, (float*)nullptr, b.att16, b.col_start, b.col_count);
    else if (bf16) launch_args(decode_cross_attention<8, __nv_bfloat16>, dim3(attn_blocks), dim3(256), 0, s, pdl_u, (const float*)b.qc, reinterpret_cast<const __nv_bfloat16*>(ckv), (int64_t)a.S, (const int*)b.nk, (const int*)b.row_start, (const float*)b.kbias_c, (int)a.n_cand, Nw, H, scale, (float*)nullptr, b.att16, b.orig);
    else decode_cross_attention<8, float><<<attn_blocks, 256, 0, s>>>(b.qc, reinterpret_cast<const float*>(ckv), a.S, b.nk, b.row_start, b.kbias_c, a.n_cand, Nw, H, scale, b.att, b.att16, b.orig);
    return check_launch(e, "decode_cross_attention", s);
}

// Launches of the decode step over the Nw rows of one wave; the residual stream is b.x (fp32) with its bf16 copy b.x16.
struct DecOps {
    mmt_engine* e; const DecBuffers& b; int64_t Nw; bool pdl_u; cudaStream_t s;
    int64_t plan() const { return b.plan_rows > 0 ? b.plan_rows : Nw; }     // rows that decide the kernel variants
    // x = LN(x + bias + sum_s part[s]) (separate kernel; fp32 mode and split-K FFN2)
    int ln(const float* part, int splits, const float* bias, const float* gamma, const float* beta) const {
        LnParams q;
        memset(&q, 0, sizeof(q));
        q.splits = splits; q.part_stride = Nw * D; q.eps = 1e-5f;
        LnGroup& g = q.g[0];
        g.part = part; g.bias = bias; g.res = b.x; g.gamma = gamma; g.beta = beta; g.out = b.x; g.out_bf16 = b.x16; g.M = (int)Nw;
        g.S_in = (int)Nw; g.stride_b = 0; g.stride_s = 1; g.off = 0;
        return launch_ln(e, q, 1, (int)Nw, s);
    }
    int gemm(const float* A, int64_t lda, const float* W, const float* bias, float* C, int N, int K, int act, int splits) const {
        GemmParams p = gemm_params(N, K, N, act);
        p.g[0].A = A; p.g[0].lda = lda; p.g[0].W = W; p.g[0].bias = bias; p.g[0].C = C; p.g[0].M = (int)Nw;
        p.splits = splits; p.part_stride = Nw * D;
        return launch_gemm(e, p, 1, (int)Nw, s, plan());
    }
    // The four attention projections of the un-fused step run on the hi term of the bf16 weight split alone, like the small-wave
    // kernel's (decode_attn keeps only the hi terms in shared memory): one weight slab per stage -> 68 KB instead of 100 KB of
    // shared memory per CTA (three resident tiles per SM instead of two), half the weight TMA bytes and MMAs.  At every wave
    // size, so that a shard decoded alone reproduces its rows of the full call bit for bit.  Measured on the golden cases:
    // worst logit error 6.37e-3 -> 6.20e-3 of the row scale, mean +12 % (profiles/r02_bf16_error_dec_proj_terms.txt).
    // MMT_DEC_PROJ_TWO_TERM=1 restores both terms.
    const __nv_bfloat16* plo(const float* w) const { return e->dec_proj_single ? nullptr : e->Wlo(w); }
    // The decoder FFN runs on the hi term of the bf16 weight split alone: measured on the 12 golden cases the lo term changes
    // the worst logit error from 5.75e-3 to 5.76e-3 of the row scale (profiles/r02_bf16_error.md) for twice the tensor work.
    // MMT_DEC_FFN_TWO_TERM=1 restores it.
    const __nv_bfloat16* dlo(const float* w) const { return e->dec_ffn_single ? nullptr : e->Wlo(w); }
    // tensor-core variants: plain projection (fp32 or bf16 out) and projection + residual + LN in place on x / x16
    int tc(const __nv_bfloat16* A, int64_t lda, const float* W, const float* bias, float* C32, __nv_bfloat16* C16, int N, int K, int act, int splits) const {
        TcGemmParams p = tc_params((int)Nw, N, K);
        p.bias = bias; p.act = act; p.out_f32 = C32; p.ld_f32 = N; p.out_b16 = C16; p.ld_b16 = N;
        p.splits = splits; p.part_stride = Nw * D;
        return launch_tc(e, p, A, lda, e->Wb(W), TC_EPI_STORE, s, plo(W), pdl_u);
    }
    int tc_ln(const __nv_bfloat16* A, int64_t lda, const float* W, const float* bias, int K, const float* gamma, const float* beta,
              const TcChain* chain = nullptr) const {
        TcGemmParams p = tc_params((int)Nw, D, K);
        p.bias = bias; p.res = b.x; p.gamma = gamma; p.beta = beta;
        p.out_f32 = b.x; p.ld_f32 = D; p.out_b16 = b.x16; p.ld_b16 = D;
        return launch_tc(e, p, A, lda, e->Wb(W), TC_EPI_LN, s, plo(W), pdl_u, chain);
    }
};

// Un-fused step, one decoder layer after its self-attention (att16 | att): x = norm1(x + out_proj(att)), then the
// cross-attention query projection of x -> qc.  decode_step and the unit hook mmt_decode_layer_tail both run this.
static int decode_self_tail_layer(const DecOps& o, const LayerW& w, bool bf16) {
    const DecBuffers& b = o.b;
    if (bf16) {
        // out-proj + LN1 and the cross-attention query projection as one launch -- for waves up to 24,576 rows: the chained
        // kernel holds 192 KB of shared memory (one CTA per SM instead of three), which costs more than the saved launch
        // once there are several tiles per SM (measured: 1383 -> 1357 us per position at 16,384 rows, 4851 -> 4901 at 65,536)
        if (o.e->use_gemm_chain && o.plan() <= 24576) {
            const TcChain ch{o.e->Wb(w.ca_in_w), o.plo(w.ca_in_w), w.ca_in_b, b.qc, D};
            MMT_TRY(o.tc_ln(b.att16, D, w.out_w, w.out_b, D, w.n1_w, w.n1_b, &ch));
        } else {
            MMT_TRY(o.tc_ln(b.att16, D, w.out_w, w.out_b, D, w.n1_w, w.n1_b));
            MMT_TRY(o.tc(b.x16, D, w.ca_in_w, w.ca_in_b, b.qc, nullptr, D, D, 0, 1));
        }
    } else {
        MMT_TRY(o.gemm(b.att, D, w.out_w, nullptr, b.part, D, D, 0, 1));
        MMT_TRY(o.ln(b.part, 1, w.out_b, w.n1_w, w.n1_b));
        MMT_TRY(o.gemm(b.x, D, w.ca_in_w, w.ca_in_b, b.qc, D, D, 0, 1));
    }
    return 0;
}

// Un-fused step, layer l after its cross attention (att16 | att): x = norm2(x + ca_out_proj(att)), then
// x = norm3(x + FFN(x)).  x2 (unit hook only; decode_step passes nullptr): receives x after norm2 where the variant stores it,
// i.e. not with the FFN prologue, which keeps it inside the FFN kernel.  decode_step and mmt_decode_layer_tail both run this.
static int decode_cross_tail_layer(const DecOps& o, const LayerW& w, int l, bool bf16, float* x2 = nullptr) {
    mmt_engine* e = o.e;
    const DecBuffers& b = o.b;
    const int M = (int)o.Nw, F = e->desc.d_ff;
    cudaStream_t s = o.s;
    auto keep_x2 = [&]() -> int {
        if (x2) MMT_CUDA(cudaMemcpyAsync(x2, b.x, (size_t)M * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
        return 0;
    };
    if (bf16) {
        const bool ffn_pro = e->use_ffn_prologue && o.plan() >= 2048;     // cross-attention out-projection + norm2 as the FFN kernel's prologue
        if (!ffn_pro) { MMT_TRY(o.tc_ln(b.att16, D, w.ca_out_w, w.ca_out_b, D, w.n2_w, w.n2_b)); MMT_TRY(keep_x2()); }
        if (o.plan() >= 2048) {
            FfnParams f = ffn_params(M, F);
            f.b1 = w.l1_b; f.bias = w.l2_b; f.res = b.x; f.gamma = w.n3_w; f.beta = w.n3_b; f.out_f32 = b.x; f.out_b16 = b.x16;
            if (getenv("MMT_FFN_DEBUG")) {     // phase stamps of the layer-3 FFN launch (printed by run_decode)
                if (!e->ffn_dbg) { MMT_CUDA(cudaMallocManaged(&e->ffn_dbg, 4096 * 16 * sizeof(long long))); memset(e->ffn_dbg, 0, 4096 * 16 * sizeof(long long)); }
                f.dbg = l == 3 ? e->ffn_dbg : nullptr;
            }
            if (ffn_pro) {
                const FfnPro pr{e->Wb(w.ca_out_w), o.plo(w.ca_out_w), w.ca_out_b, w.n2_w, w.n2_b, b.x};
                MMT_TRY(launch_ffn(e, f, b.att16, D, e->Wb(w.l1_w), o.dlo(w.l1_w), e->Wb(w.l2_w), o.dlo(w.l2_w), TC_EPI_LN, s, o.pdl_u, &pr));
            } else
            MMT_TRY(launch_ffn(e, f, b.x16, D, e->Wb(w.l1_w), o.dlo(w.l1_w), e->Wb(w.l2_w), o.dlo(w.l2_w), TC_EPI_LN, s, o.pdl_u));
        } else {   // few rows: split F over the grid, reduce the partials in the LayerNorm kernel
            FfnParams f = ffn_params(M, F);
            f.b1 = w.l1_b; f.splits = MAX_SPLITS; f.out_f32 = b.part; f.part_stride = o.Nw * D;
            if ((int64_t)f.splits * o.Nw > b.part_rows) MMT_FAIL("decode: FFN partial buffer too small for this wave (plan_decoder)");
            MMT_TRY(launch_ffn(e, f, b.x16, D, e->Wb(w.l1_w), o.dlo(w.l1_w), e->Wb(w.l2_w), o.dlo(w.l2_w), TC_EPI_STORE, s, o.pdl_u));
            MMT_TRY(o.ln(b.part, f.splits, w.l2_b, w.n3_w, w.n3_b));
        }
    } else {
        MMT_TRY(o.gemm(b.att, D, w.ca_out_w, nullptr, b.part, D, D, 0, 1));
        MMT_TRY(o.ln(b.part, 1, w.ca_out_b, w.n2_w, w.n2_b));
        MMT_TRY(keep_x2());
        MMT_TRY(o.gemm(b.x, D, w.l1_w, w.l1_b, b.h, F, D, 1, 1));
        int splits = pick_splits((int)o.plan(), D, F);
        if ((int64_t)splits * o.Nw > b.part_rows) MMT_FAIL("decode: FFN partial buffer too small for this wave (plan_decoder)");
        MMT_TRY(o.gemm(b.h, F, w.l2_w, nullptr, b.part, D, F, 0, splits));
        MMT_TRY(o.ln(b.part, splits, w.l2_b, w.n3_w, w.n3_b));
    }
    return 0;
}

// A wave (or lane) planned for `rows` sequences takes the fused row-local step (MMT_FUSED_DECODE_ROWS)
static bool fused_wave(const mmt_engine* e, int64_t rows) { return e->fused_decode_rows > 0 && rows <= e->fused_decode_rows; }

static int decode_step(mmt_engine* e, const DecodeRun& r, int64_t n0, int64_t Nw, int Bmw, DecBuffers& b, bool bf16, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    const mmt_decode_args& a = *r.a;
    const int H = d.n_heads, dh = D / H;
    const int pps = (a.max_len + PAGE_TOKENS - 1) / PAGE_TOKENS;
    const int64_t R = (int64_t)Bmw * a.S;
    const float scale = 1.0f / sqrtf((float)dh);
    const int* step = b.ctl;
    const int64_t N_total = (int64_t)a.Bm * a.n_cand;
    const int64_t ldn = r.ldn >= 0 ? r.ldn : N_total;
    const int M = (int)Nw;

    // Small batches: every decoder operation except the FFN is local to one sequence, so two
    // fused kernels per layer replace the chain of projection / attention / LayerNorm launches
    // (kernels_decode.cuh); the previous layer's FFN2 split-K partials + norm3 are folded into the
    // next kernel's prologue (the sampler's for the last layer).
    const int64_t P = b.plan_rows > 0 ? b.plan_rows : Nw;     // a compacted wave keeps the variants of its starting size
    const bool fused = fused_wave(e, P);
    const bool pdl = fused && e->use_pdl && !e->profiling;
    // un-fused tensor-core step: the same attribute through the chain of 31 launches (every kernel of the chain waits with
    // griddepcontrol.wait before it touches its predecessor's output; the LayerNorm-only kernel has no hook and is launched plainly)
    // Only for moderate waves: measured 50.2 -> 45.2 ms for a beam search over 2560 slots, but 1426 -> 1473 us per position at
    // 16,384 sequences, where the early-scheduled CTAs take SM resources from a predecessor that is throughput-bound.
    const bool pdl_u = !fused && bf16 && e->use_pdl && !e->profiling && P <= e->pdl_rows;
    const DecOps o{e, b, Nw, pdl_u, s};
    int ffn_splits = 1;
    if (fused) {
        if (dh != 8 || H != DA_H) MMT_FAIL("decoder must have 16 heads of dim 8");
        if (!e->da_dbg && getenv("MMT_DA_DEBUG")) {
            MMT_CUDA(cudaMallocManaged(&e->da_dbg, 4096 * 16 * sizeof(long long)));
            memset(e->da_dbg, 0, 4096 * 16 * sizeof(long long));
        }
        if (!e->da_ready) {
            MMT_CUDA(cudaFuncSetAttribute(decode_attn<8, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, DA_SMEM_BYTES));
            MMT_CUDA(cudaFuncSetAttribute(decode_attn<8, __nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, DA_SMEM_BYTES));
            MMT_CUDA(cudaFuncSetAttribute(decode_attn<8, __nv_bfloat16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DA_SMEM_BYTES_CL));
            e->da_ready = true;
        }
        unsigned blocks = (unsigned)((Nw + DA_R - 1) / DA_R);
        // tensor-core mode: the FFN runs inside decode_attn, as clusters of DA_CL CTAs (kernels_decode.cuh)
        const bool cl_ffn = bf16 && e->use_cluster_ffn && d.d_ff == DA_FF;
        if (cl_ffn) blocks = (blocks + DA_CL - 1) / DA_CL * DA_CL;
        // bf16: F/64 = 32 chunks over (splits x M/128) CTAs -- enough splits to cover the SMs
        ffn_splits = pick_splits(M, D, d.d_ff);
        if (bf16) { ffn_splits = 32; while (ffn_splits > 1 && (int64_t)(ffn_splits / 2) * ((M + 127) / 128) >= e->sm_count) ffn_splits /= 2; }
        if (bf16 && e->ffn_splits_override > 0) ffn_splits = e->ffn_splits_override;
        if (!cl_ffn && (int64_t)ffn_splits * Nw > b.part_rows) MMT_FAIL("decode: FFN partial buffer too small for this wave (plan_decoder)");
        if (cl_ffn) ffn_splits = 0;
        for (int l = 0; l < d.n_dec_layers; ++l) {
            const LayerW& w = e->dec[l];
            DecAttnParams q;
            memset(&q, 0, sizeof(q));
            if (l == 0) {
                if (r.trg) { q.tokens = r.trg + n0; q.tok_shift = 0; }
                else { q.tokens = r.tokens + n0; q.tok_shift = 1; }
                q.sos = 3; q.ldn = ldn; q.E_tok = e->W("embed_trg.weight"); q.E_pos = e->W("pe_trg.weight"); q.vocab = d.vocab;
            } else {
                const LayerW& pw = e->dec[l - 1];
                q.x_in = b.x;
                if (!cl_ffn) { q.part = b.part; q.splits = ffn_splits; q.part_stride = Nw * D; q.pbias = pw.l2_b; q.pgamma = pw.n3_w; q.pbeta = pw.n3_b; }
            }
            if (cl_ffn) {
                MMT_TRY(tc_init(e));
                MMT_TRY(make_tmap(&q.tmW1, e->Wb(w.l1_w), d.d_ff, D, D));
                MMT_TRY(make_tmap(&q.tmW2, e->Wb(w.l2_w), D, d.d_ff, d.d_ff));
                q.b1 = w.l1_b; q.b2 = w.l2_b; q.n3_w = w.n3_w; q.n3_b = w.n3_b; q.x_out = b.x;
            }
            q.in_w = w.in_w; q.in_b = w.in_b; q.out_w = w.out_w; q.out_b = w.out_b; q.n1_w = w.n1_w; q.n1_b = w.n1_b;
            q.kv_pool = layer_pool(b, l); q.block_table = b.block_table; q.pps = pps;
            if (!q.kv_pool) MMT_FAIL("decode: fused step without layer-0 cache pages (run_decode planned every wave on the layer-0 table)");
            q.step = step;
            q.in_w16 = e->Wb(w.in_w); q.out_w16 = e->Wb(w.out_w); q.cq_w16 = e->Wb(w.ca_in_w); q.co_w16 = e->Wb(w.ca_out_w);
            q.cq_w = w.ca_in_w; q.cq_b = w.ca_in_b; q.co_w = w.ca_out_w; q.co_b = w.ca_out_b; q.n2_w = w.n2_w; q.n2_b = w.n2_b;
            q.ckv = b.cross_kv + (size_t)l * 2 * R * D * b.kv_esz; q.rows_total = a.S;
            q.nk = b.nk; q.row_start = b.row_start; q.kbias_c = b.kbias_c; q.n_cand = a.n_cand;
            q.x2 = b.x; q.x2_16 = bf16 ? b.x16 : nullptr; q.M = Nw; q.scale = scale; q.eps = 1e-5f;
            q.dbg = (e->da_dbg && l == 3) ? e->da_dbg : nullptr;
            prof_pre(e, s);
            const bool pdl_l = pdl && !(l == 0 && r.serial_first);
            if (cl_ffn) launch_kernel_cluster(decode_attn<8, __nv_bfloat16, true>, dim3(blocks), dim3(DA_THREADS), DA_SMEM_BYTES_CL, s, pdl_l, DA_CL, q);
            else if (bf16) launch_kernel(decode_attn<8, __nv_bfloat16>, dim3(blocks), dim3(DA_THREADS), DA_SMEM_BYTES, s, pdl_l, q);
            else launch_kernel(decode_attn<8, float>, dim3(blocks), dim3(DA_THREADS), DA_SMEM_BYTES, s, pdl_l, q);
            MMT_TRY(check_launch(e, "decode_attn", s));
            if (cl_ffn) continue;
            if (bf16) {
                FfnParams f = ffn_params(M, d.d_ff);
                f.b1 = w.l1_b; f.splits = ffn_splits; f.out_f32 = b.part; f.part_stride = Nw * D;
                f.dbg = (e->da_dbg && l == 3) ? e->da_dbg + 2048 * 16 : nullptr;
                MMT_TRY(launch_ffn(e, f, b.x16, D, e->Wb(w.l1_w), o.dlo(w.l1_w), e->Wb(w.l2_w), o.dlo(w.l2_w), TC_EPI_STORE, s, pdl));
            } else {
                MMT_TRY(o.gemm(b.x, D, w.l1_w, w.l1_b, b.h, d.d_ff, D, 1, 1));
                MMT_TRY(o.gemm(b.h, d.d_ff, w.l2_w, nullptr, b.part, D, d.d_ff, 0, ffn_splits));
            }
        }
    } else {
        // layer 0 on the position x token table (b.hist, see run_decode): the embedding's bf16 copy has no reader (it was the
        // layer-0 projection's operand), the token goes to the history instead
        const bool l0_table = b.hist != nullptr;
        __nv_bfloat16* x16 = l0_table ? nullptr : b.x16;
        prof_pre(e, s);
        if (r.trg) launch_args(decode_embed, dim3((unsigned)((Nw + 3) / 4)), dim3(128), 0, s, pdl_u, r.trg + n0, 0, 3, Nw, ldn, e->W("embed_trg.weight"), e->W("pe_trg.weight"), (int)d.vocab, step, b.x, x16, b.orig, b.hist, b.hist_ld);
        else launch_args(decode_embed, dim3((unsigned)((Nw + 3) / 4)), dim3(128), 0, s, pdl_u, (const int64_t*)(r.tokens + n0), 1, 3, Nw, ldn, e->W("embed_trg.weight"), e->W("pe_trg.weight"), (int)d.vocab, step, b.x, x16, b.orig, b.hist, b.hist_ld);
        MMT_TRY(check_launch(e, "decode_embed", s));

        for (int l = 0; l < d.n_dec_layers; ++l) {
            const LayerW& w = e->dec[l];
            const char* ckv = b.cross_kv + (size_t)l * 2 * R * D * b.kv_esz;
            MMT_TRY(decode_self_attention_layer(e, w, b, layer_pool(b, l), pps, Nw, bf16, pdl_u, s, l == 0 && l0_table));
            MMT_TRY(decode_self_tail_layer(o, w, bf16));
            MMT_TRY(decode_cross_attention_layer(e, a, b, ckv, Nw, Bmw, bf16, pdl_u, s));
            MMT_TRY(decode_cross_tail_layer(o, w, l, bf16));
        }
    }
    SampleParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.x = b.x; sp.W = e->W("fc_out.weight"); sp.b = e->W("fc_out.bias"); sp.V = d.vocab; sp.N = Nw; sp.ldn = ldn;
    sp.temperature = a.temperature; sp.mode = r.mode;
    const int64_t Nrng = r.per_memory_rng ? a.n_cand : (a.N_total > 0 ? a.N_total : N_total);
    sp.rng = rng_geom(e, a.philox_seed, a.philox_offset, Nrng * d.vocab, a.rng_sm_count, a.rng_max_threads_per_sm, &sp.rng_inc);
    sp.rng_dev = b.rng_state;
    sp.seq_index_base = a.seq_index_base + n0;      // waves and lanes start at column boundaries: n0 is a multiple of n_cand
    if (r.per_memory_rng) { sp.rng_cand = a.n_cand; sp.rng_col_steps = a.max_len; }
    sp.tokens = r.tokens ? r.tokens + n0 : nullptr; sp.probs = r.probs ? r.probs + n0 : nullptr;
    sp.logits = r.logits ? r.logits + n0 * d.vocab : nullptr;
    sp.target = r.target ? r.target + n0 : nullptr; sp.target_prob = r.target_prob ? r.target_prob + n0 : nullptr;
    sp.ctl.step = b.ctl; sp.ctl.done_ctas = b.ctl + 1; sp.ctl.nonpad = (r.mode == 0) ? b.ctl + 8 : nullptr;
    sp.advance = 1;
    if (b.eos_len) { sp.orig = b.orig; sp.eos_len = b.eos_len; sp.live = b.ctl + 8 + 128; sp.eos = r.eos; }
    if (r.ctl_temp) {      // the lane's columns start at column n0 / n_cand
        const int64_t c0 = n0 / a.n_cand;
        sp.ctl_temp = r.ctl_temp + c0; sp.ctl_topk = r.ctl_topk + c0; sp.ctl_topp = r.ctl_topp + c0; sp.ctl_cand = a.n_cand;
    }
    if (fused && ffn_splits > 0) {   // norm3 of the last layer over the FFN2 partials (the cluster variant has applied it)
        const LayerW& pw = e->dec[d.n_dec_layers - 1];
        sp.part = b.part; sp.splits = ffn_splits; sp.part_stride = Nw * D;
        sp.pbias = pw.l2_b; sp.pgamma = pw.n3_w; sp.pbeta = pw.n3_b; sp.eps = 1e-5f;
    }
    return launch_sample(e, sp, P, r.ctl_temp != nullptr, pdl || pdl_u, s);
}

// Sequences a decode wave may hold (MMT_MAX_WAVE_SEQS, else by precision and device memory; see run_decode).
static int64_t max_wave_sequences(const mmt_engine* e, int precision) {
    return e->max_wave_seqs > 0 ? e->max_wave_seqs
                                : (precision == MMT_PREC_BF16 ? (int64_t)e->sm_count * (e->total_mem >= ((size_t)128 << 30) ? 8 : 4) * 128 : 32768);
}

// ---------------------------------------------------------------------------
// step graphs and lanes of the decode drivers
// ---------------------------------------------------------------------------
// A decode step is the same kernel sequence at every position (the step counter and page parity live on the device), so
// the drivers capture a group of U consecutive steps once into a CUDA graph (programmatic-dependent-launch edges included)
// and replay it.  The group spans 1..4 lanes, independent parts of a wave whose steps are parallel branches of the graph.
// A graph with a key -- the caller's tag and every value its nodes bake in -- is kept in the engine's graph cache (4
// entries, the least recently used evicted) and serves later calls with the same key; one without belongs to the
// StepGraph and is destroyed with it.
struct StepGraph {
    mmt_engine* e;
    int lanes, U;
    std::vector<uint64_t> key;        // empty: not cached
    cudaGraphExec_t exec = nullptr;
    int64_t launches = 0;             // kernel launches one replay stands for
    StepGraph(mmt_engine* e_, int lanes_, int U_) : e(e_), lanes(lanes_), U(U_) {}
    StepGraph(const StepGraph&) = delete;
    StepGraph& operator=(const StepGraph&) = delete;
    ~StepGraph() { if (key.empty() && exec) cudaGraphExecDestroy(exec); }

    // look the graph up under `k` and the values every step graph bakes in
    void find(std::vector<uint64_t> k) {
        for (uint64_t v : {(uint64_t)lanes, (uint64_t)U, (uint64_t)(uintptr_t)e->arena, (uint64_t)e->arena_bytes,
                           (uint64_t)e->fused_decode_rows, (uint64_t)e->use_pdl, (uint64_t)(uintptr_t)e->da_dbg}) k.push_back(v);
        key = std::move(k);
        for (auto& c : e->graph_cache)
            if (c.key == key) { exec = c.exec; launches = c.launches_per_group; c.stamp = ++e->graph_cache_clock; return; }
    }

    // (re)capture U steps of the lanes in `active` (bit i: lane i); step(i, stream) enqueues one step of lane i
    int capture(unsigned active, const std::function<int(int, cudaStream_t)>& step) {
        if (key.empty() && exec) cudaGraphExecDestroy(exec);
        exec = nullptr;
        for (int i = 0; i < lanes; ++i) {     // capture-only streams: the caller's stream may be the legacy default stream
            if (!e->cap_stream[i]) MMT_CUDA(cudaStreamCreateWithFlags(&e->cap_stream[i], cudaStreamNonBlocking));
            if (!e->lane_ev[i]) MMT_CUDA(cudaEventCreateWithFlags(&e->lane_ev[i], cudaEventDisableTiming));
        }
        const int64_t l0 = e->launches;
        MMT_CUDA(cudaStreamBeginCapture(e->cap_stream[0], cudaStreamCaptureModeRelaxed));
        int rc = 0;
        cudaError_t fe = cudaSuccess;
        if (lanes > 1) {                      // fork the other lanes' branches off the capture origin
            fe = cudaEventRecord(e->lane_ev[0], e->cap_stream[0]);
            for (int i = 1; i < lanes && fe == cudaSuccess; ++i) if (active >> i & 1) fe = cudaStreamWaitEvent(e->cap_stream[i], e->lane_ev[0], 0);
        }
        for (int u = 0; u < U && !rc && fe == cudaSuccess; ++u)
            for (int i = 0; i < lanes && !rc; ++i) if (active >> i & 1) rc = step(i, e->cap_stream[i]);
        for (int i = 1; i < lanes && fe == cudaSuccess; ++i) {   // join
            if (!(active >> i & 1)) continue;
            fe = cudaEventRecord(e->lane_ev[i], e->cap_stream[i]);
            if (fe == cudaSuccess) fe = cudaStreamWaitEvent(e->cap_stream[0], e->lane_ev[i], 0);
        }
        cudaGraph_t graph = nullptr;
        cudaError_t ce = cudaStreamEndCapture(e->cap_stream[0], &graph);
        launches = e->launches - l0;
        e->launches = l0;
        if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
        if (fe != cudaSuccess) { if (graph) cudaGraphDestroy(graph); MMT_FAIL(std::string("step graph lane fork/join failed: ") + cudaGetErrorString(fe)); }
        if (ce != cudaSuccess) MMT_FAIL(std::string("step graph capture failed: ") + cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(&exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { exec = nullptr; MMT_FAIL(std::string("cudaGraphInstantiate failed: ") + cudaGetErrorString(ce)); }
        if (!key.empty()) {
            if (e->graph_cache.size() >= 4) {
                size_t lru = 0;
                for (size_t i = 1; i < e->graph_cache.size(); ++i) if (e->graph_cache[i].stamp < e->graph_cache[lru].stamp) lru = i;
                cudaGraphExecDestroy(e->graph_cache[lru].exec);
                e->graph_cache.erase(e->graph_cache.begin() + lru);
            }
            e->graph_cache.push_back({key, exec, launches, ++e->graph_cache_clock});
        }
        return 0;
    }

    int replay(cudaStream_t s) {
        MMT_CUDA(cudaGraphLaunch(exec, s));
        e->launches += launches;
        return 0;
    }
};

// steps per graph group: the largest divisor of T up to MMT_GRAPH_STEPS
static int step_group(const mmt_engine* e, int T) {
    int U = 1;
    for (int u = 2; u <= e->graph_steps; ++u) if (T % u == 0) U = u;
    return U;
}

// Lanes of the decode wave of spectra [wb0, wb0 + Bmw): lane i takes the wave's spectra [i * Bm_lane, (i + 1) * Bm_lane);
// lanes left empty by a short wave are dropped.  Returns the number of lanes.
constexpr int MAX_LANES = 4;
struct Lane { int b0, Bm; int64_t n0, Nw; };
static int wave_lanes(int wb0, int Bmw, int NL, int Bm_lane, int n_cand, Lane* lane) {
    int nl = 0;
    for (int i = 0; i < NL; ++i) {
        const int lo = std::min(i * Bm_lane, Bmw), hi = std::min(lo + Bm_lane, Bmw);
        if (hi > lo) lane[nl++] = {wb0 + lo, hi - lo, (int64_t)(wb0 + lo) * n_cand, (int64_t)(hi - lo) * n_cand};
    }
    return nl;
}

// MMT_FFN_DEBUG / MMT_DA_DEBUG: print the phase timestamps the kernels of the last decode recorded (SM cycles).
// `rows`: sequences of that decode's first wave.
static int print_debug_phases(mmt_engine* e, int64_t rows, cudaStream_t s) {
    if (e->ffn_dbg) {  // un-fused FFN launch of layer 3, last position
        MMT_CUDA(cudaStreamSynchronize(s));
        for (int bshow : {0, 64, 127}) {
            const long long* d = e->ffn_dbg + bshow * 16;
            fprintf(stderr, "ffn_fused_tc<LN> CTA %d: setup %lld | first acc1 %lld | first convert %lld | chunks 8..15:", bshow, d[1] - d[0], d[2] - d[1], d[3] - d[2]);
            for (int i = 9; i <= 15; ++i) fprintf(stderr, " %lld", d[i] - d[i - 1]);
            fprintf(stderr, " | start->acc2 %lld | tmem->stage %lld | LN rows %lld | total %lld\n", d[4] - d[0], d[5] - d[4], d[6] - d[5], d[7] - d[0]);
        }
    }
    if (e->da_dbg) {   // the last decode_attn launch of layer 3
        MMT_CUDA(cudaStreamSynchronize(s));
        const int blocks = (int)std::min<int64_t>(4096, (rows + DA_R - 1) / DA_R);
        for (int bshow : {0, blocks / 2, blocks - 1}) {
            fprintf(stderr, "decode_attn phases, CTA %d:", bshow);
            const int last = e->da_dbg[bshow * 16 + 14] ? 14 : 10;     // cluster variant: 10 gather | 11 GEMM1 | 12 GEMM2 | 13 scatter | 14 norm3
            for (int i = 1; i <= last; ++i) fprintf(stderr, " %lld", e->da_dbg[bshow * 16 + i] - e->da_dbg[bshow * 16 + i - 1]);
            fprintf(stderr, "  total %lld\n", e->da_dbg[bshow * 16 + last] - e->da_dbg[bshow * 16]);
        }
        for (int bshow : {1, blocks / 2}) {
            const long long* d = e->da_dbg + (1024 + bshow) * 16;
            fprintf(stderr, "decode_attn warp 5, CTA %d: self [K+scores %lld | V+acc %lld | reduce %lld | sync %lld]  cross [loop %lld | reduce %lld | sync %lld]\n", bshow,
                    d[1] - d[0], d[2] - d[1], d[3] - d[2], d[4] - d[3], d[6] - d[5], d[7] - d[6], d[8] - d[7]);
        }
        for (int bshow : {0, 33}) {
            const long long* d = e->da_dbg + (2048 + bshow) * 16;
            fprintf(stderr, "ffn_fused phases, CTA %d:", bshow);
            for (int i = 1; i <= 7; ++i) fprintf(stderr, " %lld", d[i] - d[i - 1]);
            fprintf(stderr, "  total %lld\n", d[7] - d[0]);
        }
    }
    return 0;
}

static int run_decode(mmt_engine* e, const DecodeRun& r, int32_t* h_steps, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    const mmt_decode_args& a = *r.a;
    if (a.Bm <= 0 || a.n_cand <= 0 || a.S <= 0) MMT_FAIL("decode: empty batch");
    if (a.max_len < 1 || a.max_len > d.max_len || a.max_len > 128) MMT_FAIL("decode: max_len must be in [1, min(128, pe_trg rows)]");
    if (r.T > a.max_len) MMT_FAIL("decode: T > max_len");
    if (!(a.temperature > 0.f) && r.mode != 2) MMT_FAIL("decode: temperature must be > 0");
    if ((a.stride_s % 4) || (a.stride_b % 4) || ((uintptr_t)a.d_memory % 16)) MMT_FAIL("decode: memory must be 16-byte aligned with strides that are multiples of 4 floats");
    const int64_t N_total = (int64_t)a.Bm * a.n_cand;
    // waves: bound the self-attention KV pool (fp32: max_len*6*2*128*4 B per sequence)
    // Sequences decoded together.  A wave's KV pool is 393 KB per sequence in bf16 (6 layers x 8 pages x 8 KB; twice that in
    // fp32), so the default is ~75,000 sequences = 29.8 GB in bf16 and 32,768 in fp32.  Larger waves amortise the ~31 kernel
    // boundaries of an un-fused step: measured 1376 -> 1214 us per position and 16,384 sequences going from waves of
    // 16,384 to 65,536 (profiles/r02_config3.md); 131,072 in one wave is within 1 % of that for twice the pool.
    // (bf16: four full rounds of 128-row tiles over the SMs -- 75,776 rows on 148 SMs, 29.8 GB of pool -- so that the
    // tile-per-CTA kernels of a full wave do not end in a partly filled round: 1024 x 128 sequences run as 592 + 432 tiles =
    // 4 + 3 rounds instead of 2 x 3.46 -> 2 x 4.)
    // (second half of round 2: EIGHT full rounds -- 151,552 rows, 59.6 GB of pool -- where the device has the memory (>= 128 GB):
    // the whole 1024 x 128 job is then one wave and 128 x 31 kernel boundaries disappear, 951 -> 940 ms per decode.)
    const int64_t max_wave_seqs = max_wave_sequences(e, a.precision);
    int Bm_wave = (int)std::max<int64_t>(1, std::min<int64_t>(a.Bm, max_wave_seqs / a.n_cand));
    const int n_waves = (a.Bm + Bm_wave - 1) / Bm_wave;
    if (a.precision != MMT_PREC_FP32 && a.precision != MMT_PREC_BF16) MMT_FAIL("decode: bad precision");
    const bool bf16 = a.precision == MMT_PREC_BF16;
    // Lanes: a small wave is a latency chain of ~13 dependent kernels per position that leaves most of the GPU
    // idle, so the wave's spectra are split into independent lanes whose chains run concurrently (parallel
    // branches of the same CUDA graph, own KV pools / step counters); every sequence is independent (SURVEY 8e).
    const int64_t Nwave = (int64_t)Bm_wave * a.n_cand;
    const bool small_wave = fused_wave(e, Nwave);
    int NL = 1;
    if (small_wave && e->use_graph && !e->profiling) {
        NL = std::min(std::min(e->decode_lanes, MAX_LANES), Bm_wave);
        while (NL > 1 && Nwave / NL < 32) --NL;
    } else if (!small_wave && bf16 && e->use_graph && !e->profiling && Nwave >= 4096) {
        // Large waves: the step alternates HBM-bound kernels (self-attention over the KV pages) with tensor-bound ones
        // (the FFN), each leaving the other resource idle.  Two lanes -- independent halves of the wave as parallel
        // branches of the step graph -- let one half's attention stream pages while the other half's FFN runs.
        NL = std::min(std::min(e->decode_lanes_large, MAX_LANES), Bm_wave);
    }
    const int Bm_lane = (Bm_wave + NL - 1) / NL;
    // Single-wave sampling runs write ids / probabilities into engine-owned staging buffers (copied to the caller's
    // tensors at the end): nothing a captured decode-step graph touches then depends on the caller's allocations, so the
    // instantiated graph is reused across calls (capture + instantiation of ~400 nodes costs ~1.2 ms with the GPU idle).
    // (A retiring call's large waves capture graphs specific to its sequences' lengths, which are not cached; its small
    // waves never compact, so their one graph is cached like the plain call's.)
    const bool retire = r.eos >= 0;
    const bool staged = e->use_graph && e->use_graph_cache && !e->profiling && n_waves == 1 && r.mode != 2 && !r.trg && (!retire || small_wave);   // forced inputs are the caller's tensor: nothing to cache across calls
    // Layer 0 on the position x token table: the un-fused bf16 step with token-major pages (the fused small-wave step and the
    // other page layouts keep the cache).  Layer 0's pages are only planned if some wave of the run is a fused one.
    bool l0_table = false, l0_pool = true;
    if (bf16 && e->use_l0_table && e->use_kv_epilogue && e->kv_tok_major && d.n_heads % 8 == 0 && d.vocab <= 256) {
        bool any_fused = false;
        for (int wb0 = 0; wb0 < a.Bm; wb0 += Bm_wave) {
            Lane lane[MAX_LANES];
            const int nl = wave_lanes(wb0, std::min(Bm_wave, a.Bm - wb0), NL, Bm_lane, a.n_cand, lane);
            for (int i = 0; i < nl; ++i) (fused_wave(e, lane[i].Nw) ? any_fused : l0_table) = true;
        }
        l0_pool = any_fused;
    }
    if (l0_table) MMT_TRY(ensure_l0_table(e, s));
    Arena ar;
    DecBuffers lb[MAX_LANES];
    int64_t* st_tokens = nullptr; float* st_probs = nullptr;
    int* eos_all = nullptr;                  // retiring call: first-<EOS> step of every sequence (max_len until it emits)
    const bool controlled = r.h_temp != nullptr;
    float *ctl_temp = nullptr, *ctl_topp = nullptr; int32_t* ctl_topk = nullptr;   // (Bm) per-column sampling controls
    MMT_TRY(plan_arena(e, ar, [&]() {
        for (int i = 0; i < NL; ++i) plan_decoder(ar, d, (int64_t)Bm_lane * a.n_cand, Bm_lane, a.S, a.max_len, lb[i], bf16, e->fused_decode_rows, 1, retire, l0_table, l0_pool);
        if (staged) { st_tokens = ar.get<int64_t>((size_t)a.max_len * N_total); st_probs = ar.get<float>((size_t)a.max_len * N_total); }
        if (retire) eos_all = ar.get<int>(N_total);
        if (controlled) { ctl_temp = ar.get<float>(a.Bm); ctl_topk = ar.get<int32_t>(a.Bm); ctl_topp = ar.get<float>(a.Bm); }
    }));
    DecodeRun rs = r;                        // the run as the kernels see it
    if (staged) { rs.tokens = st_tokens; rs.probs = r.probs ? st_probs : nullptr; }
    if (controlled) {     // device copies at fixed arena addresses: a cached decode graph serves calls with other values
        MMT_CUDA(cudaMemcpyAsync(ctl_temp, r.h_temp, (size_t)a.Bm * sizeof(float), cudaMemcpyHostToDevice, s));
        MMT_CUDA(cudaMemcpyAsync(ctl_topk, r.h_topk, (size_t)a.Bm * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        MMT_CUDA(cudaMemcpyAsync(ctl_topp, r.h_topp, (size_t)a.Bm * sizeof(float), cudaMemcpyHostToDevice, s));
        rs.ctl_temp = ctl_temp; rs.ctl_topk = ctl_topk; rs.ctl_topp = ctl_topp;
    }
    const int pps = (a.max_len + PAGE_TOKENS - 1) / PAGE_TOKENS;
    // Per-step counts the host reads back, ctl[8 + t] of every lane: non-<PAD> picks (greedy) and, in a retiring call,
    // the sequences not finished after step t.  Greedy stop_on_all_pad ends the call after the first step at which every
    // sequence of every wave has emitted <PAD> (validate_generate_MMT_v15_4.py:763); a retiring call ends after the first
    // step that leaves none unfinished.
    const bool pad_stop = r.mode == 0 && a.stop_on_all_pad;
    const bool counts = retire || pad_stop;
    std::vector<int64_t> nonpad_total(r.T, 0), live_total(r.T, 0), rows_at(r.T, 0);
    if (retire) {
        fill_i32<<<(unsigned)((N_total + 255) / 256), 256, 0, s>>>(eos_all, N_total, a.max_len);
        MMT_CUDA(cudaGetLastError());
    }
    if (counts) for (int i = 0; i < 2; ++i) if (!e->poll_ev[i]) MMT_CUDA(cudaEventCreateWithFlags(&e->poll_ev[i], cudaEventDisableTiming));
    if (bf16) MMT_TRY(tc_init(e));
    for (int wb0 = 0; wb0 < a.Bm; wb0 += Bm_wave) {
        Lane lane[MAX_LANES];
        const int nl = wave_lanes(wb0, std::min(Bm_wave, a.Bm - wb0), NL, Bm_lane, a.n_cand, lane);
        int64_t rows[MAX_LANES];              // rows of each lane's wave (a retiring call's large waves shrink)
        for (int i = 0; i < nl; ++i) {
            DecBuffers& b = lb[i];
            MMT_CUDA(cudaMemsetAsync(b.ctl, 0, (8 + 256) * sizeof(int), s));
            set_u64x2<<<1, 1, 0, s>>>(b.rng_state, a.philox_seed, a.philox_offset);
            prof_pre(e, s);
            init_block_table<<<(unsigned)((lane[i].Nw * pps + 255) / 256), 256, 0, s>>>(b.block_table, lane[i].Nw, pps);
            MMT_TRY(check_launch(e, "init_block_table", s));
            MMT_TRY(decode_prepare_wave(e, a, lane[i].b0, lane[i].Bm, b, bf16, s));
            if (retire) { b.plan_rows = lane[i].Nw; b.orig = b.col_start = b.col_count = nullptr; b.eos_len = eos_all + lane[i].n0; }
            rows[i] = lane[i].Nw;
        }
        auto step = [&](int i, cudaStream_t cs) { return decode_step(e, rs, lane[i].n0, rows[i], lane[i].Bm, lb[i], bf16, cs); };
        auto active = [&]() { unsigned m = 0; for (int i = 0; i < nl; ++i) if (rows[i] > 0) m |= 1u << i; return m; };
        // a retiring call's groups are 8 positions (a shorter last group runs without the graph)
        int U = retire ? std::min(r.T, 8) : step_group(e, r.T);
        StepGraph graph(e, nl, U);
        if (staged) {
            uint32_t tbits; memcpy(&tbits, &a.temperature, 4);
            graph.find({0xDEC, (uint64_t)r.mode, (uint64_t)r.T, (uint64_t)(r.probs != nullptr), (uint64_t)a.S, (uint64_t)a.Bm,
                        (uint64_t)a.n_cand, (uint64_t)a.max_len, tbits, (uint64_t)a.precision, (uint64_t)a.seq_index_base,
                        (uint64_t)a.N_total, (uint64_t)a.rng_sm_count, (uint64_t)a.rng_max_threads_per_sm, (uint64_t)r.per_memory_rng,
                        (uint64_t)r.eos, (uint64_t)controlled});   // controls: their presence, never their values
        }
        if (e->use_graph && !e->profiling && !graph.exec) MMT_TRY(graph.capture(active(), step));
        else if (!graph.exec && !retire) U = 1;
        // Polls: after a group is enqueued, its per-step counts are copied back (poll n) and the host reads poll n - 1,
        // whose groups the GPU has finished while it runs this one, so the loop never drains the stream.  A retiring wave
        // polls every group, the single wave of a greedy stop_on_all_pad call every ~16 steps (a multiple of U); other
        // waves do not poll, and only a call that needs the counts reads them once the wave is done.
        const bool wave_pad_stop = pad_stop && n_waves == 1;
        const int poll_every = retire ? U : wave_pad_stop ? (U >= 16 ? U : (16 / U) * U) : 0;
        int n_polls = 0, polled_t[2] = {0, 0};
        const int32_t* cnt = nullptr;         // the poll the host read last: lane i's nonpad at [i * 256 + t], live at [i * 256 + 128 + t]
        auto post = [&](int t) -> int {
            for (int i = 0; i < nl; ++i)
                MMT_CUDA(cudaMemcpyAsync(e->h_pinned + (n_polls & 1) * 1024 + i * 256, lb[i].ctl + 8, 256 * sizeof(int), cudaMemcpyDeviceToHost, s));
            MMT_CUDA(cudaEventRecord(e->poll_ev[n_polls & 1], s));
            polled_t[n_polls & 1] = t;
            ++n_polls;
            return 0;
        };
        auto read = [&](int k) -> int {
            MMT_CUDA(cudaEventSynchronize(e->poll_ev[k & 1]));
            cnt = e->h_pinned + (k & 1) * 1024;
            return 0;
        };
        auto total = [&](int field, int q) { int64_t v = 0; for (int i = 0; i < nl; ++i) v += cnt[i * 256 + field + q]; return v; };
        bool stop = false;
        for (int t = 0; t < r.T && !stop;) {
            const int n = std::min(U, r.T - t);
            if (graph.exec && n == U) MMT_TRY(graph.replay(s));
            else for (int q = 0; q < n; ++q) for (int i = 0; i < nl; ++i) if (rows[i] > 0) MMT_TRY(step(i, s));
            for (int q = t; q < t + n; ++q) for (int i = 0; i < nl; ++i) rows_at[q] += rows[i];
            t += n;
            if (!poll_every || (t % poll_every && t < r.T)) continue;
            MMT_TRY(post(t));
            if (n_polls < 2 || t >= r.T) continue;
            MMT_TRY(read(n_polls - 2));
            const int tp = polled_t[n_polls & 1] - 1;      // the last step poll n - 2 covers
            for (int q = 0; q <= tp && !stop; ++q) stop = (retire && total(128, q) == 0) || (wave_pad_stop && total(0, q) == 0);
            if (stop || !retire) continue;
            // A large lane whose live rows after step tp are at most 7/8 of its wave is compacted to those rows before the
            // next group (rows finished during the group the GPU runs ride along once, masked), and the group graph is
            // captured again for the smaller wave.  Small (fused) waves are latency chains that fewer rows do not shorten:
            // they only stop once all have finished.
            bool changed = false;
            for (int i = 0; i < nl; ++i) {
                const int64_t live = cnt[i * 256 + 128 + tp];
                if (rows[i] == 0 || fused_wave(e, lb[i].plan_rows) || live * 8 > rows[i] * 7) continue;
                DecBuffers& b = lb[i];
                if (live > 0) {
                    int* orig_new = b.orig == b.rt_orig[0] ? b.rt_orig[1] : b.rt_orig[0];
                    MMT_CUDA(cudaMemsetAsync(b.rt_col_count, 0, lane[i].Bm * sizeof(int), s));
                    prof_pre(e, s);
                    retire_scan<<<1, 1024, 0, s>>>(b.orig, b.eos_len, rows[i], tp, b.rt_src);
                    MMT_TRY(check_launch(e, "retire_scan", s));
                    prof_pre(e, s);
                    retire_gather<<<(unsigned)((live + 255) / 256), 256, 0, s>>>(b.rt_src, b.orig, b.block_table, pps, live, a.n_cand, orig_new,
                                                                                 b.rt_bt, b.rt_col_start, b.rt_col_count);
                    MMT_TRY(check_launch(e, "retire_gather", s));
                    std::swap(b.block_table, b.rt_bt);
                    b.orig = orig_new; b.col_start = b.rt_col_start; b.col_count = b.rt_col_count;
                }
                rows[i] = live;
                changed = true;
            }
            if (changed && graph.exec) MMT_TRY(graph.capture(active(), step));
        }
        if (counts) {     // the wave's counts: the poll that stopped it, else one taken after its last step
            if (!stop) {
                if (!poll_every) MMT_TRY(post(r.T));
                MMT_TRY(read(n_polls - 1));
            }
            for (int q = 0; q < r.T; ++q) { nonpad_total[q] += total(0, q); live_total[q] += total(128, q); }
        }
    }
    if (staged) {
        MMT_CUDA(cudaMemcpyAsync(r.tokens, st_tokens, (size_t)r.T * N_total * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
        if (r.probs) MMT_CUDA(cudaMemcpyAsync(r.probs, st_probs, (size_t)r.T * N_total * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    // steps a wave never launched count zero: a wave that stopped early ends the call no later than its stop
    int steps_done = r.T;
    for (int q = 0; q < r.T; ++q)
        if ((retire && live_total[q] == 0) || (pad_stop && nonpad_total[q] == 0)) { steps_done = q + 1; break; }
    if (retire) {
        prof_pre(e, s);
        retire_fill<<<(unsigned)(((int64_t)r.T * N_total + 255) / 256), 256, 0, s>>>(r.tokens, r.probs, r.T, N_total, eos_all, steps_done, r.len);
        MMT_TRY(check_launch(e, "retire_fill", s));
        if (r.h_rows) for (int q = 0; q < r.T; ++q) r.h_rows[q] = rows_at[q];
    }
    if (h_steps) *h_steps = steps_done;
    return print_debug_phases(e, std::min<int64_t>(N_total, max_wave_seqs), s);
}

// Wave loop shared by the batched beam search (run_beam) and the stochastic beam search (run_sbs): the K slots of every
// memory column are K rows of one KV-cached wave; per step one decoder step over all slots (forced-token mode,
// single-row token / logit buffers), then the search's `select` kernel and beam_copy_pages (kernels_beam.cuh).  The
// per-step kernel sequence is position independent (step counter and page parity live on the device), so groups of
// steps replay as one CUDA graph.  `select` adds the slots still open after step t to ctl[8 + t]: once a step leaves
// none open, the remaining steps are fixed points and the wave stops at the next poll.
struct BeamWave { int b0, Bmw; int64_t n0, Nw; };
struct BeamLoop {
    int K, T, Bm_wave;
    DecBuffers* b;
    float* logits; int64_t* cur_tok; int *copy_src, *copy_dst;
    std::function<int(const BeamWave&, cudaStream_t)> init;     // state of the wave's slots (before the memory projection)
    std::function<int(const BeamWave&, cudaStream_t)> select;   // one selection step (captured)
    std::function<int(const BeamWave&, cudaStream_t)> finish;   // optional: after the wave's last step
    // optional: a tag and every value the step graph of a wave bakes in besides those StepGraph::find adds -> the graph
    // is kept in the engine's graph cache and serves later calls with the same key
    std::function<void(const BeamWave&, std::vector<uint64_t>&)> graph_key;
};

static int beam_wave_loop(mmt_engine* e, const mmt_decode_args& a, bool bf16, const BeamLoop& L, int32_t* h_steps, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    DecBuffers& b = *L.b;
    const int K = L.K, T = L.T;
    const int n_waves = (a.Bm + L.Bm_wave - 1) / L.Bm_wave;
    if (bf16) MMT_TRY(tc_init(e));
    int steps_max = 0;
    for (int wv = 0; wv < n_waves; ++wv) {
        BeamWave w;
        w.b0 = wv * L.Bm_wave; w.Bmw = std::min(L.Bm_wave, a.Bm - w.b0);
        w.n0 = (int64_t)w.b0 * K; w.Nw = (int64_t)w.Bmw * K;
        MMT_CUDA(cudaMemsetAsync(b.ctl, 0, (8 + 256) * sizeof(int), s));
        MMT_TRY(L.init(w, s));
        MMT_TRY(decode_prepare_wave(e, a, w.b0, w.Bmw, b, bf16, s));
        DecodeRun r;
        r.a = &a; r.mode = 2; r.trg = L.cur_tok; r.T = T; r.tokens = nullptr; r.probs = nullptr; r.logits = L.logits;
        r.ldn = 0; r.serial_first = true;
        // the wave addresses its slots from 0: pools of a smaller last wave keep the planned (larger) layer stride
        const size_t page_bytes = (size_t)2 * PAGE_TOKENS * D * b.kv_esz;
        auto one_step = [&](cudaStream_t cs) -> int {
            MMT_TRY(decode_step(e, r, 0, w.Nw, w.Bmw, b, bf16, cs));
            MMT_TRY(L.select(w, cs));
            prof_pre(e, cs);
            beam_copy_pages<<<dim3((unsigned)w.Nw, d.n_dec_layers), 256, 0, cs>>>(b.kv_pool, (size_t)b.pool_pages * page_bytes, (int)page_bytes, L.copy_src, L.copy_dst);
            MMT_TRY(check_launch(e, "beam_copy_pages", cs));
            return 0;
        };
        int U = step_group(e, T);
        StepGraph graph(e, 1, U);
        if (L.graph_key && e->use_graph && e->use_graph_cache && !e->profiling) {
            std::vector<uint64_t> key;
            L.graph_key(w, key);
            graph.find(std::move(key));
        }
        if (e->use_graph && !e->profiling && !graph.exec) MMT_TRY(graph.capture(1, [&](int, cudaStream_t cs) { return one_step(cs); }));
        else if (!graph.exec) U = 1;
        // a synchronous poll every ~16 steps (a multiple of U)
        const int poll_every = U >= 16 ? U : (16 / U) * U;
        int steps_done = T;
        for (int t = 0; t < T; t += U) {
            if (graph.exec) MMT_TRY(graph.replay(s));
            else MMT_TRY(one_step(s));
            const int done = t + U;
            if (done < T && done % poll_every == 0) {
                MMT_CUDA(cudaMemcpyAsync(e->h_pinned, b.ctl + 8, done * sizeof(int), cudaMemcpyDeviceToHost, s));
                MMT_CUDA(cudaStreamSynchronize(s));
                bool stop = false;
                for (int q = 0; q < done; ++q) if (e->h_pinned[q] == 0) { steps_done = q + 1; stop = true; break; }
                if (stop) break;
            }
        }
        if (L.finish) MMT_TRY(L.finish(w, s));
        steps_max = std::max(steps_max, steps_done);
        if (n_waves > 1) MMT_CUDA(cudaStreamSynchronize(s));   // the next wave reuses the pools
    }
    if (h_steps) *h_steps = steps_max;
    return 0;
}

// Batched beam search (reference validate_generate_MMT_v15_4.py:995-1086) on beam_wave_loop: beam_init + beam_select.
static int run_beam(mmt_engine* e, const mmt_decode_args& a0, int K, int T, int eos, int64_t* d_seq, int32_t* d_len,
                    double* d_score, float* d_probs, int32_t* h_steps, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    if (a0.Bm <= 0 || a0.S <= 0) MMT_FAIL("beam: empty batch");
    if (K < 1 || K > BEAM_MAX || K > d.vocab) MMT_FAIL("beam: beam_size must be in [1, min(32, vocab)]");
    if (T < 1 || T > d.max_len || T > 128) MMT_FAIL("beam: gen_len must be in [1, min(128, pe_trg rows)]");
    if (eos < 0 || eos >= d.vocab) MMT_FAIL("beam: bad <EOS> id");
    if ((a0.stride_s % 4) || (a0.stride_b % 4) || ((uintptr_t)a0.d_memory % 16)) MMT_FAIL("beam: memory must be 16-byte aligned with strides that are multiples of 4 floats");
    if (a0.precision != MMT_PREC_FP32 && a0.precision != MMT_PREC_BF16) MMT_FAIL("beam: bad precision");
    const bool bf16 = a0.precision == MMT_PREC_BF16;
    mmt_decode_args a = a0;
    a.n_cand = K; a.max_len = T; a.temperature = 1.f; a.sampling = MMT_SAMPLE_GREEDY; a.stop_on_all_pad = 0;
    const int pps = (T + PAGE_TOKENS - 1) / PAGE_TOKENS;
    BeamLoop L;
    L.K = K; L.T = T;
    L.Bm_wave = (int)std::max<int64_t>(1, std::min<int64_t>(a.Bm, 8192 / K));
    const int64_t Nw_max = (int64_t)L.Bm_wave * K;
    Arena ar;
    DecBuffers b;
    L.b = &b;
    MMT_TRY(plan_arena(e, ar, [&]() {
        plan_decoder(ar, d, Nw_max, L.Bm_wave, a.S, T, b, bf16, e->fused_decode_rows, 2);
        L.logits = ar.get<float>((size_t)Nw_max * d.vocab);
        L.cur_tok = ar.get<int64_t>((size_t)Nw_max);
        L.copy_src = ar.get<int>((size_t)Nw_max); L.copy_dst = ar.get<int>((size_t)Nw_max);
    }));
    auto params = [&](const BeamWave& w) {
        BeamParams bp;
        memset(&bp, 0, sizeof(bp));
        bp.logits = L.logits; bp.V = d.vocab; bp.K = K; bp.T = T; bp.eos = eos; bp.pps = pps; bp.Nw = w.Nw; bp.step = b.ctl;
        bp.score = d_score + w.n0; bp.len = d_len + w.n0; bp.hist = d_seq + w.n0 * (T + 1); bp.probs = d_probs + w.n0 * T;
        bp.cur_tok = L.cur_tok; bp.block_table = b.block_table; bp.copy_src = L.copy_src; bp.copy_dst = L.copy_dst; bp.unfinished = b.ctl + 8;
        return bp;
    };
    L.init = [&](const BeamWave& w, cudaStream_t cs) -> int {
        prof_pre(e, cs);
        beam_init<<<(unsigned)((w.Nw + 255) / 256), 256, 0, cs>>>(params(w), 3);
        return check_launch(e, "beam_init", cs);
    };
    L.select = [&](const BeamWave& w, cudaStream_t cs) -> int {
        prof_pre(e, cs);
        beam_select<<<w.Bmw, 256, 0, cs>>>(params(w));
        return check_launch(e, "beam_select", cs);
    };
    return beam_wave_loop(e, a, bf16, L, h_steps, s);
}

// Stochastic beam search (kernels_sbs.cuh) on beam_wave_loop.  Waves: two page parities, so at most half the decode
// wave of the precision (max_wave_sequences / 2 slots), in whole columns.  Slot state lives in the arena (both
// parities) and the column temperatures are copied there before the first step, so a wave's step graph -- kept in the
// graph cache -- serves later calls with other temperatures, generator states and outputs; sbs_finish writes the
// caller's tensors after the wave's last step.
static int run_sbs(mmt_engine* e, const mmt_decode_args& a0, const float* h_temp, int eos, int64_t* d_tokens, float* d_probs,
                   int32_t* d_len, double* d_log_prob, double* d_key, int32_t* h_steps, cudaStream_t s) {
    const mmt_model_desc& d = e->desc;
    const int K = a0.n_cand, T = a0.max_len, V = d.vocab;
    const bool bf16 = a0.precision == MMT_PREC_BF16;
    mmt_decode_args a = a0;
    a.temperature = 1.f; a.sampling = MMT_SAMPLE_GREEDY; a.stop_on_all_pad = 0; a.seq_index_base = 0; a.N_total = 0;
    const int pps = (T + PAGE_TOKENS - 1) / PAGE_TOKENS;
    BeamLoop L;
    L.K = K; L.T = T;
    L.Bm_wave = (int)std::max<int64_t>(1, std::min<int64_t>(a.Bm, max_wave_sequences(e, a.precision) / 2 / K));
    const int64_t Nw_max = (int64_t)L.Bm_wave * K;
    Arena ar;
    DecBuffers b;
    L.b = &b;
    double *phi[2], *key[2]; int* len[2]; uint8_t* hist[2]; float* probs[2]; float* temp = nullptr;
    MMT_TRY(plan_arena(e, ar, [&]() {
        plan_decoder(ar, d, Nw_max, L.Bm_wave, a.S, T, b, bf16, e->fused_decode_rows, 2);
        L.logits = ar.get<float>((size_t)Nw_max * V);
        L.cur_tok = ar.get<int64_t>((size_t)Nw_max);
        L.copy_src = ar.get<int>((size_t)Nw_max); L.copy_dst = ar.get<int>((size_t)Nw_max);
        for (int i = 0; i < 2; ++i) {
            phi[i] = ar.get<double>((size_t)Nw_max); key[i] = ar.get<double>((size_t)Nw_max); len[i] = ar.get<int>((size_t)Nw_max);
            hist[i] = ar.get<uint8_t>((size_t)Nw_max * T); probs[i] = ar.get<float>((size_t)Nw_max * T);
        }
        temp = ar.get<float>((size_t)a.Bm);
    }));
    MMT_CUDA(cudaFuncSetAttribute(sbs_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sbs_smem_bytes(SBS_MAX, VOCAB_MAX)));
    MMT_CUDA(cudaMemcpyAsync(temp, h_temp, (size_t)a.Bm * sizeof(float), cudaMemcpyHostToDevice, s));
    uint64_t rng_inc;      // the generator state comes from b.rng_state
    const RngGeom rng = rng_geom(e, 0, 0, (int64_t)K * V, a.rng_sm_count, a.rng_max_threads_per_sm, &rng_inc);
    auto params = [&](const BeamWave& w) {
        SbsParams sp;
        memset(&sp, 0, sizeof(sp));
        sp.logits = L.logits; sp.V = V; sp.K = K; sp.T = T; sp.eos = eos; sp.pps = pps; sp.Nw = w.Nw; sp.step = b.ctl;
        sp.temp = temp + w.b0;
        sp.rng = rng; sp.rng_inc = rng_inc;
        sp.rng_dev = b.rng_state;
        sp.col_base = a0.seq_index_base / K + w.b0;
        for (int i = 0; i < 2; ++i) { sp.phi[i] = phi[i]; sp.key[i] = key[i]; sp.len[i] = len[i]; sp.hist[i] = hist[i]; sp.probs[i] = probs[i]; }
        sp.cur_tok = L.cur_tok; sp.block_table = b.block_table; sp.copy_src = L.copy_src; sp.copy_dst = L.copy_dst; sp.unfinished = b.ctl + 8;
        return sp;
    };
    L.init = [&](const BeamWave& w, cudaStream_t cs) -> int {
        set_u64x2<<<1, 1, 0, cs>>>(b.rng_state, a0.philox_seed, a0.philox_offset);
        prof_pre(e, cs);
        sbs_init<<<(unsigned)((w.Nw + 255) / 256), 256, 0, cs>>>(params(w), 3);
        return check_launch(e, "sbs_init", cs);
    };
    L.select = [&](const BeamWave& w, cudaStream_t cs) -> int {
        prof_pre(e, cs);
        sbs_select<<<w.Bmw, SBS_THREADS, sbs_smem_bytes(K, V), cs>>>(params(w));
        return check_launch(e, "sbs_select", cs);
    };
    L.finish = [&](const BeamWave& w, cudaStream_t cs) -> int {
        prof_pre(e, cs);
        sbs_finish<<<(unsigned)((w.Nw * T + 255) / 256), 256, 0, cs>>>(params(w), w.n0, (int64_t)a.Bm * K, d_tokens, d_probs, d_len, d_log_prob, d_key);
        return check_launch(e, "sbs_finish", cs);
    };
    L.graph_key = [&](const BeamWave& w, std::vector<uint64_t>& k) {
        for (uint64_t v : {(uint64_t)0x5B5, (uint64_t)K, (uint64_t)T, (uint64_t)eos, (uint64_t)a.S, (uint64_t)w.Bmw, (uint64_t)a.precision,
                           (uint64_t)(a0.seq_index_base / K + w.b0), (uint64_t)rng.threads, rng_inc, (uint64_t)w.b0}) k.push_back(v);
    };
    return beam_wave_loop(e, a, bf16, L, h_steps, s);
}

}  // namespace mmt

// ===========================================================================
// C ABI
// ===========================================================================
using namespace mmt;

extern "C" {

int32_t mmt_abi_version(void) { return MMT_ABI_VERSION; }
const char* mmt_last_error(void) { return g_last_error.c_str(); }

static int check_desc(const mmt_model_desc* d) {
    if (!d) MMT_FAIL("null model desc");
    if (d->d_model != D) MMT_FAIL("only hidden_size 128 is supported");
    if (d->n_heads != 16 || d->n_heads_cross < 1 || (D % d->n_heads_cross)) MMT_FAIL("unsupported head counts");
    if (d->vocab > VOCAB_MAX || d->vocab < 1) MMT_FAIL("vocab must be <= 64");
    if (d->max_len > 128 || d->max_len < 1) MMT_FAIL("max_len must be <= 128");
    if (d->d_ff % 64 || d->ir_bins % 4) MMT_FAIL("d_ff must be a multiple of 64 and ir_bins of 4");
    return 0;
}

int32_t mmt_weight_count(const mmt_model_desc* desc) { if (check_desc(desc)) return -1; return (int32_t)build_registry(*desc).slots.size(); }
const char* mmt_weight_name(const mmt_model_desc* desc, int32_t i) {
    static thread_local std::string name;
    if (check_desc(desc)) return nullptr;
    Registry r = build_registry(*desc);
    if (i < 0 || i >= (int)r.slots.size()) return nullptr;
    name = r.slots[i].name;
    return name.c_str();
}
int64_t mmt_weight_numel(const mmt_model_desc* desc, int32_t i) {
    if (check_desc(desc)) return -1;
    Registry r = build_registry(*desc);
    return (i < 0 || i >= (int)r.slots.size()) ? -1 : r.slots[i].numel;
}
int64_t mmt_weight_offset(const mmt_model_desc* desc, int32_t i) {
    if (check_desc(desc)) return -1;
    Registry r = build_registry(*desc);
    return (i < 0 || i >= (int)r.slots.size()) ? -1 : r.slots[i].off;
}
int64_t mmt_weight_total(const mmt_model_desc* desc) { if (check_desc(desc)) return -1; return build_registry(*desc).total; }

int32_t mmt_create(const mmt_model_desc* desc, const float* h_weights, int64_t n_floats, int32_t device, mmt_engine** out) {
    if (!out) MMT_FAIL("null out");
    *out = nullptr;
    MMT_TRY(check_desc(desc));
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) MMT_FAIL("no CUDA device: this engine has no CPU fallback");
    if (device < 0 || device >= ndev) MMT_FAIL("bad device index");
    cudaDeviceProp prop;
    MMT_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) MMT_FAIL(std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) + "; this library is built for sm_100a (B200) only");
    MMT_CUDA(cudaSetDevice(device));
    mmt_engine* e = new mmt_engine();
    e->desc = *desc; e->device = device; e->sm_count = prop.multiProcessorCount; e->max_threads_per_sm = prop.maxThreadsPerMultiProcessor; e->total_mem = prop.totalGlobalMem;
    e->reg = build_registry(*desc);
    if (getenv("MMT_NO_GRAPH")) e->use_graph = false;
    if (getenv("MMT_NO_PDL")) e->use_pdl = false;
    if (getenv("MMT_NO_GRAPH_CACHE")) e->use_graph_cache = false;
    if (const char* v = getenv("MMT_GRAPH_STEPS")) e->graph_steps = std::max(1, atoi(v));
    if (getenv("MMT_NO_ENC_STREAMS")) e->use_enc_streams = false;
    if (const char* v = getenv("MMT_DECODE_LANES")) e->decode_lanes = std::max(1, atoi(v));
    if (getenv("MMT_DENSE_ENCODER")) e->use_compact = false;
    if (getenv("MMT_NO_TC_ATTENTION")) e->use_tc_attention = false;
    if (getenv("MMT_TC5_ATTENTION")) e->use_tc5_attention = true;
    if (const char* v = getenv("MMT_FFN_SPLITS")) { int k = atoi(v); if (k == 1 || k == 2 || k == 4 || k == 8 || k == 16 || k == 32) e->ffn_splits_override = k; }
    if (getenv("MMT_TC_ATTENTION_FP32")) e->tc_attention_fp32 = true;
    if (const char* v = getenv("MMT_FUSED_DECODE_ROWS")) e->fused_decode_rows = atoi(v);
    if (getenv("MMT_DEC_FFN_TWO_TERM")) e->dec_ffn_single = false;
    if (getenv("MMT_DEC_PROJ_TWO_TERM")) e->dec_proj_single = false;
    if (const char* v = getenv("MMT_PDL_ROWS")) e->pdl_rows = atoi(v);
    if (getenv("MMT_NO_GEMM_CHAIN")) e->use_gemm_chain = false;
    if (getenv("MMT_NO_FFN_WIDE")) e->use_ffn_wide = false;
    if (getenv("MMT_NO_KV_EPILOGUE")) e->use_kv_epilogue = false;
    if (getenv("MMT_NO_L0_TABLE")) e->use_l0_table = false;
    if (getenv("MMT_KV_HEAD_MAJOR")) e->kv_tok_major = false;
    if (getenv("MMT_CLUSTER_FFN")) e->use_cluster_ffn = true;
    if (getenv("MMT_NO_FFN_PROLOGUE")) e->use_ffn_prologue = false;
    if (getenv("MMT_ENC_FFN_SINGLE")) e->enc_ffn_single = true;
    if (const char* v = getenv("MMT_DECODE_LANES_LARGE")) e->decode_lanes_large = std::max(1, atoi(v));
    if (const char* v = getenv("MMT_MAX_WAVE_SEQS")) e->max_wave_seqs = std::max(1, atoi(v));     // 0 / unset: by precision
    if (n_floats != e->reg.total) { delete e; MMT_FAIL("weight blob has " + std::to_string(n_floats) + " floats, expected " + std::to_string(build_registry(*desc).total)); }
    auto fail = [&](const std::string& m) { mmt_destroy(e); g_last_error = m; return 1; };
    if (cudaMalloc(&e->w32, n_floats * sizeof(float)) != cudaSuccess) return fail("cudaMalloc weights failed");
    if (cudaMalloc(&e->w16, n_floats * sizeof(__nv_bfloat16)) != cudaSuccess) return fail("cudaMalloc bf16 weights failed");
    if (cudaMemcpy(e->w32, h_weights, n_floats * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) return fail("weight H2D copy failed");
    if (cudaMalloc(&e->w16lo, n_floats * sizeof(__nv_bfloat16)) != cudaSuccess) return fail("cudaMalloc bf16 weights (low term) failed");
    f32_to_bf16_split<<<(unsigned)((n_floats + 255) / 256), 256>>>(e->w32, n_floats, e->w16, e->w16lo);
    if (cudaDeviceSynchronize() != cudaSuccess) return fail(std::string("bf16 weight conversion failed: ") + cudaGetErrorString(cudaGetLastError()));
    if (cudaMallocHost(&e->h_pinned, 2048 * sizeof(int32_t)) != cudaSuccess) return fail("cudaMallocHost failed");
    for (int k = 0; k < 6; ++k) {
        e->enc[k].resize(desc->n_enc_layers);
        for (int l = 0; l < desc->n_enc_layers; ++l) fill_layer(e, e->enc[k][l], std::string(kEncNames[k]) + ".layers." + std::to_string(l), false);
    }
    e->dec.resize(desc->n_dec_layers);
    for (int l = 0; l < desc->n_dec_layers; ++l) fill_layer(e, e->dec[l], "decoder.layers." + std::to_string(l), true);
    *out = e;
    return 0;
}

void mmt_destroy(mmt_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    if (e->w32) cudaFree(e->w32);
    if (e->w16) cudaFree(e->w16);
    if (e->w16lo) cudaFree(e->w16lo);
    if (e->arena) cudaFree(e->arena);
    if (e->l0_qtab) cudaFree(e->l0_qtab);
    if (e->l0_kvtab) cudaFree(e->l0_kvtab);
    if (e->h_pinned) cudaFreeHost(e->h_pinned);
    for (auto& c : e->graph_cache) cudaGraphExecDestroy(c.exec);
    for (int i = 0; i < 5; ++i) if (e->enc_stream[i]) cudaStreamDestroy(e->enc_stream[i]);
    for (int i = 0; i < 6; ++i) if (e->enc_ev[i]) cudaEventDestroy(e->enc_ev[i]);
    for (int i = 0; i < 4; ++i) { if (e->cap_stream[i]) cudaStreamDestroy(e->cap_stream[i]); if (e->lane_ev[i]) cudaEventDestroy(e->lane_ev[i]); }
    for (int i = 0; i < 2; ++i) if (e->poll_ev[i]) cudaEventDestroy(e->poll_ev[i]);
    if (e->last_use) cudaEventDestroy(e->last_use);
    delete e;
}

int32_t mmt_memory_len(const mmt_model_desc* desc, uint32_t mode_bits) {
    if (check_desc(desc)) return -1;
    return mode_layout(*desc, mode_bits).S_total;
}
int32_t mmt_mask_is_float(uint32_t mode_bits) {
    for (int m = 0; m < 4; ++m) if (!((mode_bits >> m) & 1)) return 1;
    return 0;
}

int32_t mmt_encode(mmt_engine* e, const mmt_spectra* in, int32_t B, uint32_t mode_bits, int32_t precision,
                   float* d_memory, float* d_embedding_src, float* d_key_bias, uint8_t* d_pad_mask,
                   float* d_fingerprint, float* d_avg_memory, void* stream) {
    if (!e || !in) MMT_FAIL("null engine / spectra");
    if (B <= 0) MMT_FAIL("encode: B must be > 0");
    if (!d_memory && !d_embedding_src) MMT_FAIL("encode: d_memory is required (or d_embedding_src alone for an embedding-only call)");
    if (!d_memory && (d_fingerprint || d_avg_memory)) MMT_FAIL("encode: fingerprint / mean need d_memory");
    if (precision != MMT_PREC_FP32 && precision != MMT_PREC_BF16) MMT_FAIL("bad precision");
    // reference constraints (SURVEY.md B.4): some NMR modality and MW must be present
    if (!(mode_bits & 0xF)) MMT_FAIL("training_mode needs at least one of 1H/13C/HSQC/COSY (the reference crashes without)");
    if (!(mode_bits & MMT_MODE_MW)) MMT_FAIL("training_mode needs MW (the reference crashes without)");
    cudaStream_t s = (cudaStream_t)stream;
    EngineCall call(e, s);
    const ModeLayout L = mode_layout(e->desc, mode_bits);
    const int chunk = 256;
    for (int b0 = 0; b0 < B; b0 += chunk) {
        int Bc = std::min(chunk, B - b0);
        // ragged path: all five spectra in training_mode (bool key-padding masks everywhere; SURVEY.md A.2, B.2)
        int rc = 2;
        if (d_memory && e->use_compact && !L.float_mask && L.present[4])
            rc = encode_chunk_compact(e, *in, b0, Bc, B, L, d_memory, d_embedding_src, d_key_bias, d_pad_mask, precision == MMT_PREC_BF16, s);
        if (rc == 1) return 1;
        if (rc == 2) MMT_TRY(encode_chunk(e, *in, b0, Bc, B, mode_bits, L, d_memory, d_embedding_src, d_key_bias, d_pad_mask, precision == MMT_PREC_BF16, s));
    }
    if (d_fingerprint || d_avg_memory) {
        Arena a;
        a.plan = false; a.base = e->arena; a.cap = e->arena_bytes; a.off = 0;
        MMT_TRY(ensure_arena(e, (size_t)B * D * sizeof(float) + 256));
        a.base = e->arena;
        float* avg = d_avg_memory ? d_avg_memory : a.get<float>((size_t)B * D);
        prof_pre(e, s);
        mean_over_sequence<<<B, 128, 0, s>>>(d_memory, L.S_total, B, avg);
        MMT_TRY(check_launch(e, "mean_over_sequence", s));
        if (d_fingerprint) {
            GemmParams p = gemm_params(e->desc.fp_size, D, e->desc.fp_size, 0);
            p.g[0].A = avg; p.g[0].lda = D; p.g[0].W = e->W("fp1.weight"); p.g[0].bias = e->W("fp1.bias"); p.g[0].C = d_fingerprint; p.g[0].M = B;
            MMT_TRY(launch_gemm(e, p, 1, B, s));
        }
    }
    return 0;
}

int32_t mmt_decode(mmt_engine* e, const mmt_decode_args* a, int64_t* d_tokens, float* d_probs, int32_t* h_steps, void* stream) {
    if (!e || !a) MMT_FAIL("null engine / args");
    if (!d_tokens) MMT_FAIL("decode: d_tokens is required");
    if (a->sampling != MMT_SAMPLE_GREEDY && a->sampling != MMT_SAMPLE_MULTINOMIAL) MMT_FAIL("bad sampling mode");
    EngineCall call(e, (cudaStream_t)stream);
    DecodeRun r;
    r.a = a; r.mode = a->sampling; r.trg = nullptr; r.T = a->max_len; r.tokens = d_tokens; r.probs = d_probs; r.logits = nullptr;
    return run_decode(e, r, h_steps, (cudaStream_t)stream);
}

int32_t mmt_decode_memory_streams(mmt_engine* e, const mmt_decode_args* a, int64_t* d_tokens, float* d_probs, int32_t* h_steps, void* stream) {
    if (!e || !a) MMT_FAIL("null engine / args");
    if (!d_tokens) MMT_FAIL("decode: d_tokens is required");
    if (a->sampling != MMT_SAMPLE_MULTINOMIAL) MMT_FAIL("mmt_decode_memory_streams: per-memory RNG streams need multinomial sampling");
    if (a->n_cand <= 0 || a->seq_index_base < 0 || a->seq_index_base % a->n_cand)
        MMT_FAIL("mmt_decode_memory_streams: seq_index_base must be a non-negative multiple of n_cand");
    EngineCall call(e, (cudaStream_t)stream);
    DecodeRun r;
    r.a = a; r.mode = a->sampling; r.trg = nullptr; r.T = a->max_len; r.tokens = d_tokens; r.probs = d_probs; r.logits = nullptr;
    r.per_memory_rng = true;
    return run_decode(e, r, h_steps, (cudaStream_t)stream);
}

int32_t mmt_decode_until_eos(mmt_engine* e, const mmt_decode_args* a, int32_t per_memory_rng, int64_t eos, int64_t* d_tokens, float* d_probs,
                             int32_t* d_len, int32_t* h_steps, int64_t* h_rows, void* stream) {
    if (!e || !a) MMT_FAIL("null engine / args");
    if (!d_tokens || !d_len) MMT_FAIL("mmt_decode_until_eos: d_tokens and d_len are required");
    if (a->sampling != MMT_SAMPLE_GREEDY && a->sampling != MMT_SAMPLE_MULTINOMIAL) MMT_FAIL("bad sampling mode");
    if (per_memory_rng) {
        if (a->sampling != MMT_SAMPLE_MULTINOMIAL) MMT_FAIL("mmt_decode_until_eos: per-memory RNG streams need multinomial sampling");
        if (a->n_cand <= 0 || a->seq_index_base < 0 || a->seq_index_base % a->n_cand)
            MMT_FAIL("mmt_decode_until_eos: seq_index_base must be a non-negative multiple of n_cand");
    }
    if (eos < 0 || eos >= e->desc.vocab) MMT_FAIL("mmt_decode_until_eos: eos must be in [0, vocab)");
    EngineCall call(e, (cudaStream_t)stream);
    DecodeRun r;
    r.a = a; r.mode = a->sampling; r.trg = nullptr; r.T = a->max_len; r.tokens = d_tokens; r.probs = d_probs; r.logits = nullptr;
    r.per_memory_rng = per_memory_rng != 0; r.eos = eos; r.len = d_len; r.h_rows = h_rows;
    return run_decode(e, r, h_steps, (cudaStream_t)stream);
}

// The caller's sampling controls for Bm columns, checked on the host, as full host arrays (absent ones: temperature
// `t_default`, top-k 0, top-p 1).
static int host_controls(const mmt_sampling_controls* c, int64_t Bm, float t_default, int V, std::vector<float>& temp,
                         std::vector<int32_t>& topk, std::vector<float>& topp, const char* who) {
    if (!c) MMT_FAIL(std::string(who) + ": sampling controls are required");
    if ((c->h_temperature || c->h_top_k || c->h_top_p) && c->count != Bm)
        MMT_FAIL(std::string(who) + ": sampling controls hold " + std::to_string(c->count) + " columns, the call has " + std::to_string(Bm));
    temp.assign(Bm, t_default); topk.assign(Bm, 0); topp.assign(Bm, 1.f);
    for (int64_t b = 0; b < Bm; ++b) {
        if (c->h_temperature) temp[b] = c->h_temperature[b];
        if (c->h_top_k) topk[b] = c->h_top_k[b];
        if (c->h_top_p) topp[b] = c->h_top_p[b];
        if (!(temp[b] > 0.f) || !std::isfinite(temp[b])) MMT_FAIL(std::string(who) + ": temperature must be > 0 and finite (column " + std::to_string(b) + ")");
        if (topk[b] < 0 || topk[b] > V) MMT_FAIL(std::string(who) + ": top_k must be in [0, vocab] (column " + std::to_string(b) + ")");
        if (!(topp[b] > 0.f && topp[b] <= 1.f)) MMT_FAIL(std::string(who) + ": top_p must be in (0, 1] (column " + std::to_string(b) + ")");
    }
    return 0;
}

int32_t mmt_decode_controlled(mmt_engine* e, const mmt_decode_args* a, int32_t per_memory_rng, int64_t eos, const mmt_sampling_controls* c,
                              int64_t* d_tokens, float* d_probs, int32_t* d_len, int32_t* h_steps, int64_t* h_rows, void* stream) {
    if (!e || !a) MMT_FAIL("null engine / args");
    if (!d_tokens) MMT_FAIL("mmt_decode_controlled: d_tokens is required");
    if (a->sampling != MMT_SAMPLE_MULTINOMIAL) MMT_FAIL("mmt_decode_controlled: sampling controls need multinomial sampling");
    if (per_memory_rng && (a->n_cand <= 0 || a->seq_index_base < 0 || a->seq_index_base % a->n_cand))
        MMT_FAIL("mmt_decode_controlled: seq_index_base must be a non-negative multiple of n_cand");
    if (eos >= 0 && (eos >= e->desc.vocab || !d_len)) MMT_FAIL("mmt_decode_controlled: eos must be in [0, vocab) and d_len given");
    if (a->Bm <= 0 || a->n_cand <= 0) MMT_FAIL("decode: empty batch");
    std::vector<float> temp, topp; std::vector<int32_t> topk;
    MMT_TRY(host_controls(c, a->Bm, a->temperature, e->desc.vocab, temp, topk, topp, "mmt_decode_controlled"));
    EngineCall call(e, (cudaStream_t)stream);
    DecodeRun r;
    r.a = a; r.mode = a->sampling; r.trg = nullptr; r.T = a->max_len; r.tokens = d_tokens; r.probs = d_probs; r.logits = nullptr;
    r.per_memory_rng = per_memory_rng != 0;
    if (eos >= 0) { r.eos = eos; r.len = d_len; r.h_rows = h_rows; }
    r.h_temp = temp.data(); r.h_topk = topk.data(); r.h_topp = topp.data();
    return run_decode(e, r, h_steps, (cudaStream_t)stream);
}

int32_t mmt_teacher_forced(mmt_engine* e, const mmt_decode_args* a, const int64_t* d_trg, int32_t T, float* d_logits, void* stream) {
    if (!e || !a || !d_trg || !d_logits) MMT_FAIL("null argument");
    if (T < 1) MMT_FAIL("T must be >= 1");
    EngineCall call(e, (cudaStream_t)stream);
    DecodeRun r;
    r.a = a; r.mode = 2; r.trg = d_trg; r.T = T; r.tokens = nullptr; r.probs = nullptr; r.logits = d_logits;
    return run_decode(e, r, nullptr, (cudaStream_t)stream);
}

int32_t mmt_beam_search(mmt_engine* e, const mmt_decode_args* a, int32_t beam_size, int32_t gen_len, int32_t eos,
                        int64_t* d_seq, int32_t* d_len, double* d_score, float* d_probs, int32_t* h_steps, void* stream) {
    if (!e || !a || !d_seq || !d_len || !d_score || !d_probs) MMT_FAIL("null argument");
    EngineCall call(e, (cudaStream_t)stream);
    return run_beam(e, *a, beam_size, gen_len, eos, d_seq, d_len, d_score, d_probs, h_steps, (cudaStream_t)stream);
}

// Column temperatures of a stochastic beam search: h_temperature (Bm) or a->temperature for every column, checked.
static int sbs_temperatures(const float* h_temperature, int64_t Bm, float t_default, std::vector<float>& temp, const char* who) {
    temp.assign(Bm, t_default);
    for (int64_t b = 0; b < Bm; ++b) {
        if (h_temperature) temp[b] = h_temperature[b];
        if (!(temp[b] > 0.f) || !std::isfinite(temp[b])) MMT_FAIL(std::string(who) + ": temperature must be > 0 and finite (column " + std::to_string(b) + ")");
    }
    return 0;
}

int32_t mmt_sample_without_replacement(mmt_engine* e, const mmt_decode_args* a, const float* h_temperature, int32_t eos,
                                       int64_t* d_tokens, float* d_probs, int32_t* d_len, double* d_log_prob, double* d_key,
                                       int32_t* h_steps, void* stream) {
    const char* who = "mmt_sample_without_replacement";
    if (!e || !a) MMT_FAIL("null engine / args");
    if (!d_tokens || !d_probs || !d_len || !d_log_prob || !d_key) MMT_FAIL(std::string(who) + ": every output is required");
    if (a->Bm <= 0 || a->S <= 0) MMT_FAIL(std::string(who) + ": empty batch");
    const int64_t K = a->n_cand;
    if (K < 1 || K > SBS_MAX) MMT_FAIL(std::string(who) + ": n_cand must be in [1, 128]");
    if (a->max_len < 1 || a->max_len > e->desc.max_len || a->max_len > 128) MMT_FAIL(std::string(who) + ": max_len must be in [1, min(128, pe_trg rows)]");
    if (eos < 0 || eos >= e->desc.vocab) MMT_FAIL(std::string(who) + ": eos must be in [0, vocab)");
    if (a->seq_index_base < 0 || a->seq_index_base % K) MMT_FAIL(std::string(who) + ": seq_index_base must be a non-negative multiple of n_cand");
    if (a->N_total < 0 || (a->N_total > 0 && (a->N_total % K || a->N_total < a->seq_index_base + a->Bm * K)))
        MMT_FAIL(std::string(who) + ": N_total must be 0 or a multiple of n_cand covering seq_index_base + Bm * n_cand");
    if ((a->stride_s % 4) || (a->stride_b % 4) || ((uintptr_t)a->d_memory % 16)) MMT_FAIL(std::string(who) + ": memory must be 16-byte aligned with strides that are multiples of 4 floats");
    if (a->precision != MMT_PREC_FP32 && a->precision != MMT_PREC_BF16) MMT_FAIL(std::string(who) + ": bad precision");
    std::vector<float> temp;
    MMT_TRY(sbs_temperatures(h_temperature, a->Bm, a->temperature, temp, who));
    EngineCall call(e, (cudaStream_t)stream);
    return run_sbs(e, *a, temp.data(), eos, d_tokens, d_probs, d_len, d_log_prob, d_key, h_steps, (cudaStream_t)stream);
}

int32_t mmt_sbs_select_step(mmt_engine* e, const float* d_logits, int32_t Bm, int32_t k, int32_t V, int32_t T, int32_t step, int32_t eos,
                            const float* h_temperature, uint64_t philox_seed, uint64_t philox_offset, int64_t seq_index_base,
                            int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                            const double* d_phi, const double* d_key, const int32_t* d_len, const uint8_t* d_hist, const float* d_probs,
                            double* d_phi_out, double* d_key_out, int32_t* d_len_out, uint8_t* d_hist_out, float* d_probs_out, float* d_p_out, void* stream) {
    const char* who = "mmt_sbs_select_step";
    if (!e || !d_logits || !d_phi || !d_key || !d_len || !d_hist || !d_probs || !d_phi_out || !d_key_out || !d_len_out || !d_hist_out || !d_probs_out || !h_temperature)
        MMT_FAIL("null argument");
    if (Bm < 1) MMT_FAIL(std::string(who) + ": empty batch");
    if (k < 1 || k > SBS_MAX) MMT_FAIL(std::string(who) + ": k must be in [1, 128]");
    if (V < 1 || V > VOCAB_MAX) MMT_FAIL(std::string(who) + ": V must be in [1, 64]");
    if (T < 1 || T > 128 || step < 0 || step >= T) MMT_FAIL(std::string(who) + ": need 1 <= T <= 128 and 0 <= step < T");
    if (eos < 0 || eos >= V) MMT_FAIL(std::string(who) + ": eos must be in [0, V)");
    if (seq_index_base < 0 || seq_index_base % k) MMT_FAIL(std::string(who) + ": seq_index_base must be a non-negative multiple of k");
    std::vector<float> temp;
    MMT_TRY(sbs_temperatures(h_temperature, Bm, 1.f, temp, who));
    EngineCall call(e, (cudaStream_t)stream);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t N = (int64_t)Bm * k;
    const int pps = (T + PAGE_TOKENS - 1) / PAGE_TOKENS;
    Arena ar;
    int* ctl = nullptr; float* d_temp = nullptr; int64_t* cur_tok = nullptr; int *bt = nullptr, *cs = nullptr, *cd = nullptr;
    MMT_TRY(plan_arena(e, ar, [&]() {
        ctl = ar.get<int>(1); d_temp = ar.get<float>(Bm); cur_tok = ar.get<int64_t>(N);
        bt = ar.get<int>(N * pps); cs = ar.get<int>(N); cd = ar.get<int>(N);
    }));
    const int t1 = step + 1;      // the step counter as the sampler leaves it
    MMT_CUDA(cudaMemcpyAsync(ctl, &t1, sizeof(int), cudaMemcpyHostToDevice, s));
    MMT_CUDA(cudaMemcpyAsync(d_temp, temp.data(), (size_t)Bm * sizeof(float), cudaMemcpyHostToDevice, s));
    MMT_CUDA(cudaMemsetAsync(bt, 0, (size_t)N * pps * sizeof(int), s));
    MMT_CUDA(cudaMemcpyAsync(d_hist_out, d_hist, (size_t)N * T, cudaMemcpyDeviceToDevice, s));
    MMT_CUDA(cudaMemcpyAsync(d_probs_out, d_probs, (size_t)N * T * sizeof(float), cudaMemcpyDeviceToDevice, s));
    SbsParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.logits = d_logits; sp.V = V; sp.K = k; sp.T = T; sp.eos = eos; sp.pps = pps; sp.Nw = N; sp.step = ctl; sp.temp = d_temp;
    sp.rng = rng_geom(e, philox_seed, philox_offset, (int64_t)k * V, rng_sm_count, rng_max_threads_per_sm, &sp.rng_inc);
    sp.col_base = seq_index_base / k;
    const int rd = step & 1, wr = rd ^ 1;
    sp.phi[rd] = const_cast<double*>(d_phi); sp.key[rd] = const_cast<double*>(d_key); sp.len[rd] = const_cast<int*>(d_len);
    sp.hist[rd] = const_cast<uint8_t*>(d_hist); sp.probs[rd] = const_cast<float*>(d_probs);
    sp.phi[wr] = d_phi_out; sp.key[wr] = d_key_out; sp.len[wr] = d_len_out; sp.hist[wr] = d_hist_out; sp.probs[wr] = d_probs_out;
    sp.cur_tok = cur_tok; sp.block_table = bt; sp.copy_src = cs; sp.copy_dst = cd; sp.p_out = d_p_out;
    MMT_CUDA(cudaFuncSetAttribute(sbs_select, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sbs_smem_bytes(SBS_MAX, VOCAB_MAX)));
    prof_pre(e, s);
    sbs_select<<<Bm, SBS_THREADS, sbs_smem_bytes(k, V), s>>>(sp);
    return check_launch(e, "sbs_select", s);
}

int32_t mmt_spectra_equal(mmt_engine* e, const mmt_spectra* a, const mmt_spectra* b, int32_t B, uint32_t mode_bits, int32_t* h_equal, void* stream) {
    if (!e || !a || !b || !h_equal) MMT_FAIL("null argument");
    if (B <= 0) MMT_FAIL("B must be > 0");
    EngineCall call(e, (cudaStream_t)stream);
    cudaStream_t s = (cudaStream_t)stream;
    const mmt_model_desc& d = e->desc;
    const int64_t P = d.pad_points;
    CompareParams p;
    memset(&p, 0, sizeof(p));
    int n = 0;
    bool missing = false;
    auto seg = [&](const void* x, const void* y, int64_t bytes) {
        if (!x || !y) { missing = true; return; }
        p.a[n] = reinterpret_cast<const unsigned char*>(x); p.b[n] = reinterpret_cast<const unsigned char*>(y); p.bytes[n] = bytes; ++n;
    };
    if (mode_bits & MMT_MODE_1H) { seg(a->d_src_1H, b->d_src_1H, B * P * 8); seg(a->d_mask_1H, b->d_mask_1H, B * P * 4); }
    if (mode_bits & MMT_MODE_13C) { seg(a->d_src_13C, b->d_src_13C, B * P * 4); seg(a->d_mask_13C, b->d_mask_13C, B * P * 4); }
    if (mode_bits & MMT_MODE_HSQC) { seg(a->d_src_HSQC, b->d_src_HSQC, B * P * 8); seg(a->d_mask_HSQC, b->d_mask_HSQC, B * P * 4); }
    if (mode_bits & MMT_MODE_COSY) { seg(a->d_src_COSY, b->d_src_COSY, B * P * 8); seg(a->d_mask_COSY, b->d_mask_COSY, B * P * 4); }
    if (mode_bits & MMT_MODE_IR) seg(a->d_src_IR, b->d_src_IR, (int64_t)B * d.ir_bins * 4);
    if (mode_bits & MMT_MODE_MF) { seg(a->d_src_MF, b->d_src_MF, B * P * 8); seg(a->d_mask_MF, b->d_mask_MF, B * P); }
    if (mode_bits & MMT_MODE_MS) { seg(a->d_src_MS, b->d_src_MS, B * P * 8); seg(a->d_mask_MS, b->d_mask_MS, B * P); }
    if (mode_bits & MMT_MODE_MW) seg(a->d_trg_MW, b->d_trg_MW, (int64_t)B * 4);
    if (missing) MMT_FAIL("spectra pointer missing for a modality in training_mode");
    p.n = n;
    MMT_TRY(ensure_arena(e, 256));
    int* flag = reinterpret_cast<int*>(e->arena);
    p.differ = flag;
    MMT_CUDA(cudaMemsetAsync(flag, 0, sizeof(int), s));
    compare_segments<<<dim3(64, n), 256, 0, s>>>(p);
    MMT_CUDA(cudaGetLastError());
    MMT_CUDA(cudaMemcpyAsync(e->h_pinned, flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    MMT_CUDA(cudaStreamSynchronize(s));
    *h_equal = e->h_pinned[0] == 0;
    return 0;
}

int32_t mmt_teacher_forced_scores(mmt_engine* e, const mmt_decode_args* a, const int64_t* d_trg_in, const int64_t* d_target, int32_t T,
                                  int64_t* d_pick, float* d_pick_prob, float* d_target_prob, void* stream) {
    if (!e || !a || !d_trg_in || !d_pick) MMT_FAIL("null argument");
    if (T < 1) MMT_FAIL("T must be >= 1");
    if (a->sampling != MMT_SAMPLE_GREEDY && a->sampling != MMT_SAMPLE_MULTINOMIAL) MMT_FAIL("bad sampling mode");
    if ((d_target == nullptr) != (d_target_prob == nullptr)) MMT_FAIL("d_target and d_target_prob go together");
    EngineCall call(e, (cudaStream_t)stream);
    mmt_decode_args a2 = *a;
    a2.stop_on_all_pad = 0;
    DecodeRun r;
    r.a = &a2; r.mode = a->sampling; r.trg = d_trg_in; r.T = T; r.tokens = d_pick; r.probs = d_pick_prob; r.logits = nullptr;
    r.target = d_target; r.target_prob = d_target_prob;
    return run_decode(e, r, nullptr, (cudaStream_t)stream);
}

uint64_t mmt_philox_increment(int64_t numel, int32_t sm_count, int32_t max_threads_per_sm) {
    return torch_rng_increment(numel, sm_count, max_threads_per_sm);
}

int32_t mmt_pack_tokens_u8(const int64_t* d_tokens, int64_t n, uint8_t* d_out, void* stream) {
    if (n <= 0) return 0;
    pack_tokens_u8<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_tokens, n, d_out);
    MMT_CUDA(cudaGetLastError());
    return 0;
}
int32_t mmt_unpack_tokens_u8(const uint8_t* d_in, int64_t n, int64_t* d_tokens, void* stream) {
    if (n <= 0) return 0;
    unpack_tokens_u8<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_in, n, d_tokens);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_pack_tokens_u8_seqmajor(const int64_t* d_tokens, int32_t T, int64_t N, uint8_t* d_out, void* stream) {
    if (N <= 0 || T <= 0) return 0;
    if (!d_tokens || !d_out) MMT_FAIL("null argument");
    pack_tokens_u8_seqmajor<<<dim3((unsigned)((N + 31) / 32), (unsigned)((T + 31) / 32)), 256, 0, (cudaStream_t)stream>>>(d_tokens, T, N, d_out);
    MMT_CUDA(cudaGetLastError());
    return 0;
}
int32_t mmt_unpack_tokens_u8_seqmajor(const uint8_t* d_in, int32_t T, int64_t N, int64_t* d_tokens, void* stream) {
    if (N <= 0 || T <= 0) return 0;
    if (!d_in || !d_tokens) MMT_FAIL("null argument");
    unpack_tokens_u8_seqmajor<<<dim3((unsigned)((N + 31) / 32), (unsigned)((T + 31) / 32)), 256, 0, (cudaStream_t)stream>>>(d_in, T, N, d_tokens);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_ingest_peaks(const double* d_values, const int64_t* d_offsets, int32_t B, int32_t cols, double div0, double div1,
                         int32_t pad_points, float* d_src, float* d_mask, void* stream) {
    if (!d_values || !d_offsets || !d_src || !d_mask) MMT_FAIL("null argument");
    if (cols != 1 && cols != 2) MMT_FAIL("ingest: cols must be 1 or 2");
    if (B <= 0 || pad_points <= 0) return 0;
    ingest_peaks<<<B, 64, 0, (cudaStream_t)stream>>>(d_values, d_offsets, cols, div0, div1, pad_points, cols == 1 ? 1 : 0, d_src, d_mask);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_ingest_ir(const double* d_values, const int64_t* d_offsets, int32_t B, int32_t bins, float* d_src_IR, void* stream) {
    if (!d_values || !d_offsets || !d_src_IR) MMT_FAIL("null argument");
    if (B <= 0 || bins <= 0) return 0;
    if (bins > 8192) MMT_FAIL("ingest: too many IR bins");
    ingest_ir<<<B, 256, (size_t)(bins + 1) * sizeof(int), (cudaStream_t)stream>>>(d_values, d_offsets, bins, d_src_IR);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_first_eos(const int64_t* d_tokens, int32_t T, int64_t N, int32_t eos, int32_t* d_len, void* stream) {
    if (!d_tokens || !d_len) MMT_FAIL("null argument");
    if (N <= 0 || T <= 0) return 0;
    first_eos_scan<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_tokens, T, N, eos, d_len);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_sample(mmt_engine* e, const float* d_x, int64_t N, float temperature, int32_t sampling,
                   uint64_t philox_seed, uint64_t philox_offset, int64_t seq_index_base, int64_t N_total,
                   int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                   int64_t* d_token, float* d_prob, float* d_logits_out, void* stream) {
    if (!e || !d_x) MMT_FAIL("null argument");
    if (N <= 0) return 0;
    EngineCall call(e, (cudaStream_t)stream);
    SampleParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.x = d_x; sp.W = e->W("fc_out.weight"); sp.b = e->W("fc_out.bias"); sp.V = e->desc.vocab; sp.N = N; sp.ldn = N;
    sp.temperature = temperature; sp.mode = sampling;
    const int64_t Nrng = N_total > 0 ? N_total : N;
    sp.rng = rng_geom(e, philox_seed, philox_offset, Nrng * sp.V, rng_sm_count, rng_max_threads_per_sm, &sp.rng_inc);
    sp.seq_index_base = seq_index_base;
    sp.tokens = d_token; sp.probs = d_prob; sp.logits = d_logits_out;
    sp.advance = 0;
    return launch_sample(e, sp, N, false, false, (cudaStream_t)stream);
}

int32_t mmt_exponential(uint64_t philox_seed, uint64_t philox_offset, int64_t elem_base, int64_t n, int64_t numel_total,
                        int32_t sm_count, int32_t max_threads_per_sm, float* d_q, void* stream) {
    if (!d_q) MMT_FAIL("null argument");
    if (n <= 0) return 0;
    if (sm_count <= 0 || max_threads_per_sm < 256 || numel_total < elem_base + n || elem_base < 0) MMT_FAIL("mmt_exponential: bad geometry");
    RngGeom g;
    g.seed = philox_seed; g.offset = philox_offset; g.numel = numel_total; g.threads = torch_rng_threads(numel_total, sm_count, max_threads_per_sm);
    exponential_fill<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(g, elem_base, n, d_q);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_sample_probs(const float* d_p, int64_t N, int32_t V, uint64_t philox_seed, uint64_t philox_offset,
                         int64_t seq_index_base, int64_t N_total, int32_t sm_count, int32_t max_threads_per_sm,
                         int64_t* d_token, void* stream) {
    if (!d_p || !d_token) MMT_FAIL("null argument");
    if (N <= 0) return 0;
    if (V < 1 || sm_count <= 0 || max_threads_per_sm < 256 || seq_index_base < 0) MMT_FAIL("mmt_sample_probs: bad geometry");
    const int64_t Nrng = N_total > 0 ? N_total : N;
    if (Nrng < seq_index_base + N) MMT_FAIL("mmt_sample_probs: N_total smaller than seq_index_base + N");
    RngGeom g;
    g.seed = philox_seed; g.offset = philox_offset; g.numel = Nrng * V; g.threads = torch_rng_threads(g.numel, sm_count, max_threads_per_sm);
    sample_from_probs<<<(unsigned)((N + 7) / 8), 256, 0, (cudaStream_t)stream>>>(d_p, N, V, g, seq_index_base, 0, 0, 0, 0, d_token);
    MMT_CUDA(cudaGetLastError());
    return 0;
}

int32_t mmt_sample_memory_streams(mmt_engine* e, const float* d_x, const float* d_p, int64_t N, int32_t n_cand, int32_t max_len,
                                  int32_t step, float temperature, uint64_t philox_seed, uint64_t philox_offset,
                                  int64_t seq_index_base, int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                                  int64_t* d_token, float* d_prob, void* stream) {
    if (!e || !d_token || (!d_x) == (!d_p)) MMT_FAIL("mmt_sample_memory_streams: give d_token and exactly one of d_x, d_p");
    if (n_cand <= 0 || max_len < 1 || step < 0 || step >= max_len) MMT_FAIL("mmt_sample_memory_streams: need n_cand >= 1 and 0 <= step < max_len");
    if (seq_index_base < 0 || seq_index_base % n_cand) MMT_FAIL("mmt_sample_memory_streams: seq_index_base must be a non-negative multiple of n_cand");
    if (N <= 0) return 0;
    EngineCall call(e, (cudaStream_t)stream);
    cudaStream_t cs = (cudaStream_t)stream;
    const int V = e->desc.vocab;
    uint64_t inc;
    const RngGeom g = rng_geom(e, philox_seed, philox_offset, (int64_t)n_cand * V, rng_sm_count, rng_max_threads_per_sm, &inc);
    if (d_p) {
        prof_pre(e, cs);
        sample_from_probs<<<(unsigned)((N + 7) / 8), 256, 0, cs>>>(d_p, N, V, g, seq_index_base, inc, n_cand, max_len, step, d_token);
        return check_launch(e, "sample_from_probs", cs);
    }
    // fused fc_out + softmax + pick at step `step`, read from a device step counter like the decode step's
    Arena ar;
    int* ctl = nullptr;
    MMT_TRY(plan_arena(e, ar, [&]() { ctl = ar.get<int>(1); }));
    MMT_CUDA(cudaMemcpyAsync(ctl, &step, sizeof(int), cudaMemcpyHostToDevice, cs));
    SampleParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.x = d_x; sp.W = e->W("fc_out.weight"); sp.b = e->W("fc_out.bias"); sp.V = V; sp.N = N; sp.ldn = N;
    sp.temperature = temperature; sp.mode = MMT_SAMPLE_MULTINOMIAL;
    sp.rng = g; sp.rng_inc = inc; sp.seq_index_base = seq_index_base; sp.rng_cand = n_cand; sp.rng_col_steps = max_len;
    sp.tokens = d_token - (int64_t)step * N; sp.probs = d_prob ? d_prob - (int64_t)step * N : nullptr;   // row `step` = the caller's
    sp.ctl.step = ctl;
    sp.advance = 0;
    return launch_sample(e, sp, N, false, false, cs);
}

int32_t mmt_sample_controlled(mmt_engine* e, const float* d_x, const float* d_p, int64_t N, int32_t n_cand, const mmt_sampling_controls* c,
                              int32_t per_memory_rng, int32_t max_len, int32_t step, uint64_t philox_seed, uint64_t philox_offset,
                              int64_t seq_index_base, int64_t N_total, int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                              int64_t* d_token, float* d_prob, float* d_logits_out, uint8_t* d_kept, void* stream) {
    if (!e || !d_token || (!d_x) == (!d_p)) MMT_FAIL("mmt_sample_controlled: give d_token and exactly one of d_x, d_p");
    if (n_cand <= 0 || max_len < 1 || step < 0 || step >= max_len) MMT_FAIL("mmt_sample_controlled: need n_cand >= 1 and 0 <= step < max_len");
    if (per_memory_rng && (seq_index_base < 0 || seq_index_base % n_cand))
        MMT_FAIL("mmt_sample_controlled: seq_index_base must be a non-negative multiple of n_cand");
    if (d_p && d_logits_out) MMT_FAIL("mmt_sample_controlled: d_logits_out needs d_x");
    const int V = e->desc.vocab;
    if (N <= 0) return 0;
    const int64_t Nrng = N_total > 0 ? N_total : N;
    if (!per_memory_rng && (seq_index_base < 0 || Nrng < seq_index_base + N)) MMT_FAIL("mmt_sample_controlled: N_total smaller than seq_index_base + N");
    const int64_t Bm = (N + n_cand - 1) / n_cand;
    std::vector<float> temp, topp; std::vector<int32_t> topk;
    MMT_TRY(host_controls(c, Bm, 1.f, V, temp, topk, topp, "mmt_sample_controlled"));
    EngineCall call(e, (cudaStream_t)stream);
    cudaStream_t cs = (cudaStream_t)stream;
    uint64_t inc;
    const RngGeom g = rng_geom(e, philox_seed, philox_offset, (per_memory_rng ? (int64_t)n_cand : Nrng) * V, rng_sm_count, rng_max_threads_per_sm, &inc);
    Arena ar;      // workspace: step counter, then the controls
    int* ctl = nullptr; float *ctl_temp = nullptr, *ctl_topp = nullptr; int32_t* ctl_topk = nullptr;
    MMT_TRY(plan_arena(e, ar, [&]() { ctl = ar.get<int>(1); ctl_temp = ar.get<float>(Bm); ctl_topk = ar.get<int32_t>(Bm); ctl_topp = ar.get<float>(Bm); }));
    MMT_CUDA(cudaMemcpyAsync(ctl_temp, temp.data(), (size_t)Bm * 4, cudaMemcpyHostToDevice, cs));
    MMT_CUDA(cudaMemcpyAsync(ctl_topk, topk.data(), (size_t)Bm * 4, cudaMemcpyHostToDevice, cs));
    MMT_CUDA(cudaMemcpyAsync(ctl_topp, topp.data(), (size_t)Bm * 4, cudaMemcpyHostToDevice, cs));
    if (d_p) {
        if (V > 64) MMT_FAIL("mmt_sample_controlled: vocab > 64");
        prof_pre(e, cs);
        sample_probs_controlled<<<(unsigned)((N + 7) / 8), 256, 0, cs>>>(d_p, N, V, g, seq_index_base, inc, per_memory_rng ? n_cand : 0, max_len, step,
                                                                          n_cand, ctl_topk, ctl_topp, d_token, d_prob, d_kept);
        return check_launch(e, "sample_probs_controlled", cs);
    }
    MMT_CUDA(cudaMemcpyAsync(ctl, &step, sizeof(int), cudaMemcpyHostToDevice, cs));
    SampleParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.x = d_x; sp.W = e->W("fc_out.weight"); sp.b = e->W("fc_out.bias"); sp.V = V; sp.N = N; sp.ldn = N;
    sp.temperature = 1.f; sp.mode = MMT_SAMPLE_MULTINOMIAL;
    sp.rng = g; sp.rng_inc = inc; sp.seq_index_base = seq_index_base;
    if (per_memory_rng) { sp.rng_cand = n_cand; sp.rng_col_steps = max_len; }
    // row `step` of each output = the caller's buffer
    sp.tokens = d_token - (int64_t)step * N; sp.probs = d_prob ? d_prob - (int64_t)step * N : nullptr;
    sp.logits = d_logits_out ? d_logits_out - (int64_t)step * N * V : nullptr;
    sp.kept = d_kept ? d_kept - (int64_t)step * N * V : nullptr;
    sp.ctl_temp = ctl_temp; sp.ctl_topk = ctl_topk; sp.ctl_topp = ctl_topp; sp.ctl_cand = n_cand;
    sp.ctl.step = ctl;
    sp.advance = 0;
    return launch_sample(e, sp, N, true, false, cs);
}

int32_t mmt_distinct_smiles(const int64_t* d_tokens, int32_t T, int64_t N, int32_t n_cand, int64_t eos,
                            const uint8_t* d_itos_bytes, const int32_t* d_itos_entries, int32_t n_itos, int32_t itos_max_bytes,
                            void* d_work, int64_t* work_bytes, int64_t* h_result, void* stream) {
    if (!work_bytes) MMT_FAIL("null argument");
    if (T < 1 || N < 1 || n_cand < 1 || N % n_cand || n_itos < 0 || itos_max_bytes < 0)
        MMT_FAIL("mmt_distinct_smiles: need T >= 1 and N a positive multiple of n_cand");
    const int64_t Bm = N / n_cand;
    int P = 2;
    while (P < 2 * n_cand) P <<= 1;
    const bool gtab = P > SMILES_SMEM_SLOTS;
    // workspace: scratch, then the output (metadata + bytes, at most every candidate's T entries of itos_max_bytes)
    auto al = [](int64_t x) { return (x + 255) & ~(int64_t)255; };
    const int64_t o_hash = 0, o_nbytes = o_hash + al(8 * N), o_didx = o_nbytes + al(8 * N), o_dbyte = o_didx + al(8 * (N + 1));
    const int64_t o_ntok = o_dbyte + al(8 * (N + 1)), o_slot = o_ntok + al(4 * N), o_mult = o_slot + al(4 * N), o_isd = o_mult + al(4 * N);
    const int64_t o_bad = o_isd + al(4 * N), o_tab = o_bad + 256, o_out = o_tab + (gtab ? al(4 * Bm * P) : 0);
    const int64_t need = o_out + 8 * (Bm + 1 + 4 * N + 1) + N * T * (int64_t)itos_max_bytes;
    if (!d_work) { *work_bytes = need; return 0; }
    if (*work_bytes < need || !d_tokens || !d_itos_entries || (!d_itos_bytes && n_itos) || !h_result)
        MMT_FAIL("mmt_distinct_smiles: workspace too small or null argument");
    cudaStream_t s = (cudaStream_t)stream;
    char* w = static_cast<char*>(d_work);
    SmilesParams p;
    p.tokens = d_tokens; p.T = T; p.N = N; p.k = n_cand; p.eos = eos;
    p.tab_bytes = d_itos_bytes; p.tab = reinterpret_cast<const int2*>(d_itos_entries); p.n_tab = n_itos; p.P = P;
    p.gtable = gtab ? reinterpret_cast<int*>(w + o_tab) : nullptr;
    p.hash = reinterpret_cast<uint64_t*>(w + o_hash); p.nbytes = reinterpret_cast<int64_t*>(w + o_nbytes);
    p.ntok = reinterpret_cast<int32_t*>(w + o_ntok); p.slot = reinterpret_cast<int32_t*>(w + o_slot);
    p.mult = reinterpret_cast<int32_t*>(w + o_mult); p.isd = reinterpret_cast<int32_t*>(w + o_isd);
    p.bad = reinterpret_cast<int64_t*>(w + o_bad);
    int64_t* didx = reinterpret_cast<int64_t*>(w + o_didx);
    int64_t* dbyte = reinterpret_cast<int64_t*>(w + o_dbyte);
    int64_t* out = reinterpret_cast<int64_t*>(w + o_out);
    MMT_CUDA(cudaMemsetAsync(p.bad, 0, 2 * sizeof(int64_t), s));
    const int threads = (int)std::min<int64_t>(1024, (n_cand + 31) / 32 * 32);
    smiles_dedup<<<(unsigned)Bm, threads, gtab ? 0 : (size_t)P * sizeof(int), s>>>(p);
    MMT_CUDA(cudaGetLastError());
    smiles_scan<<<1, 1024, 0, s>>>(p.isd, p.nbytes, N, didx, dbyte);
    MMT_CUDA(cudaGetLastError());
    smiles_emit<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(p, didx, dbyte, Bm, out);
    MMT_CUDA(cudaGetLastError());
    int64_t tot[4];
    MMT_CUDA(cudaMemcpyAsync(tot, didx + N, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    MMT_CUDA(cudaMemcpyAsync(tot + 1, dbyte + N, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    MMT_CUDA(cudaMemcpyAsync(tot + 2, p.bad, 2 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    MMT_CUDA(cudaStreamSynchronize(s));
    h_result[0] = tot[0];                                    // distinct strings
    h_result[1] = tot[1];                                    // bytes of the distinct strings
    h_result[2] = o_out;                                     // output offset in d_work ...
    h_result[3] = 8 * (Bm + 1 + 4 * tot[0] + 1) + tot[1];   // ... and size
    h_result[4] = tot[2];                                    // 1: an id before <EOS> has no itos entry ...
    h_result[5] = tot[3];                                    // ... this one
    return 0;
}

int32_t mmt_linear(mmt_engine* e, const float* d_A, const float* d_W, const float* d_bias, float* d_C,
                   int64_t M, int32_t N, int32_t K, int32_t act, int32_t precision, void* stream) {
    if (!e || !d_A || !d_W || !d_C) MMT_FAIL("null argument");
    if (K % 4) MMT_FAIL("K must be a multiple of 4");
    if (M > 0x7fffffff) MMT_FAIL("M too large");
    EngineCall call(e, (cudaStream_t)stream);
    cudaStream_t cs = (cudaStream_t)stream;
    if (precision == MMT_PREC_BF16) {   // convert the operands to bf16 in the workspace, then one tcgen05 GEMM
        if (K % TC_BK || N % 4) MMT_FAIL("mmt_linear bf16: K must be a multiple of 64 and N of 4");
        const size_t nA = (size_t)M * K, nW = (size_t)N * K;
        const size_t bA = (nA * 2 + 255) & ~size_t(255), bW = (nW * 2 + 255) & ~size_t(255);
        MMT_TRY(ensure_arena(e, bA + 2 * bW + 512));
        __nv_bfloat16* A16 = reinterpret_cast<__nv_bfloat16*>(e->arena);
        __nv_bfloat16* W16 = reinterpret_cast<__nv_bfloat16*>(e->arena + bA);
        __nv_bfloat16* W16lo = reinterpret_cast<__nv_bfloat16*>(e->arena + bA + bW);
        f32_to_bf16<<<(unsigned)((nA + 255) / 256), 256, 0, cs>>>(d_A, (int64_t)nA, A16);
        f32_to_bf16_split<<<(unsigned)((nW + 255) / 256), 256, 0, cs>>>(d_W, (int64_t)nW, W16, W16lo);
        MMT_CUDA(cudaGetLastError());
        TcGemmParams p = tc_params((int)M, N, K);
        p.bias = d_bias; p.act = act; p.out_f32 = d_C; p.ld_f32 = N;
        return launch_tc(e, p, A16, K, W16, TC_EPI_STORE, cs, W16lo);
    }
    if (precision != MMT_PREC_FP32) MMT_FAIL("bad precision");
    GemmParams p = gemm_params(N, K, N, act);
    p.g[0].A = d_A; p.g[0].lda = K; p.g[0].W = d_W; p.g[0].bias = d_bias; p.g[0].C = d_C; p.g[0].M = (int)M;
    return launch_gemm(e, p, 1, (int)M, cs);
}

int32_t mmt_ffn(mmt_engine* e, const float* d_x, const float* d_w1, const float* d_b1, const float* d_w2, const float* d_b2,
                const float* d_gamma, const float* d_beta, float* d_out, int64_t M, int32_t F, int32_t splits, int32_t weight_terms, void* stream) {
    if (weight_terms != 1 && weight_terms != 2) MMT_FAIL("mmt_ffn: weight_terms must be 1 or 2");
    if (!e || !d_x || !d_w1 || !d_b1 || !d_w2 || !d_b2 || !d_gamma || !d_beta || !d_out) MMT_FAIL("null argument");
    if (M <= 0) return 0;
    if (M > 0x7fffffff) MMT_FAIL("M too large");
    EngineCall call(e, (cudaStream_t)stream);
    cudaStream_t cs = (cudaStream_t)stream;
    if (splits < 1) splits = 1;
    const size_t nX = (size_t)M * D, nW = (size_t)F * D;
    auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t bX = al(nX * 2), bW = al(nW * 2), bP = al((size_t)splits * nX * 4);
    MMT_TRY(ensure_arena(e, bX + 4 * bW + bP + 512));
    char* base = e->arena;
    __nv_bfloat16* X16 = reinterpret_cast<__nv_bfloat16*>(base);
    __nv_bfloat16* W1h = reinterpret_cast<__nv_bfloat16*>(base + bX);
    __nv_bfloat16* W1l = reinterpret_cast<__nv_bfloat16*>(base + bX + bW);
    __nv_bfloat16* W2h = reinterpret_cast<__nv_bfloat16*>(base + bX + 2 * bW);
    __nv_bfloat16* W2l = reinterpret_cast<__nv_bfloat16*>(base + bX + 3 * bW);
    float* part = reinterpret_cast<float*>(base + bX + 4 * bW);
    f32_to_bf16<<<(unsigned)((nX + 255) / 256), 256, 0, cs>>>(d_x, (int64_t)nX, X16);
    f32_to_bf16_split<<<(unsigned)((nW + 255) / 256), 256, 0, cs>>>(d_w1, (int64_t)nW, W1h, W1l);
    f32_to_bf16_split<<<(unsigned)((nW + 255) / 256), 256, 0, cs>>>(d_w2, (int64_t)nW, W2h, W2l);
    MMT_CUDA(cudaGetLastError());
    FfnParams p = ffn_params((int)M, F);
    p.b1 = d_b1; p.splits = splits;
    if (splits == 1) {
        p.bias = d_b2; p.res = d_x; p.gamma = d_gamma; p.beta = d_beta; p.out_f32 = d_out;
        return launch_ffn(e, p, X16, D, W1h, weight_terms == 2 ? W1l : nullptr, W2h, weight_terms == 2 ? W2l : nullptr, TC_EPI_LN, cs);
    }
    p.out_f32 = part; p.part_stride = (int64_t)nX;
    MMT_TRY(launch_ffn(e, p, X16, D, W1h, weight_terms == 2 ? W1l : nullptr, W2h, weight_terms == 2 ? W2l : nullptr, TC_EPI_STORE, cs));
    LnParams q;
    memset(&q, 0, sizeof(q));
    q.splits = p.splits; q.part_stride = (int64_t)nX; q.eps = 1e-5f;
    LnGroup& g = q.g[0];
    g.part = part; g.bias = d_b2; g.res = d_x; g.gamma = d_gamma; g.beta = d_beta; g.out = d_out; g.M = (int)M;
    g.S_in = (int)M; g.stride_b = 0; g.stride_s = 1; g.off = 0;
    return launch_ln(e, q, 1, (int)M, cs);
}

int32_t mmt_decode_self_attention(mmt_engine* e, int32_t layer, const float* d_x, int64_t N, int32_t T, int32_t precision,
                                  float* d_out, void* stream) {
    if (!e || !d_x || !d_out) MMT_FAIL("null argument");
    const mmt_model_desc& d = e->desc;
    if (layer < 0 || layer >= d.n_dec_layers) MMT_FAIL("mmt_decode_self_attention: layer out of range");
    if (N <= 0 || N > 0x7fffffff) MMT_FAIL("mmt_decode_self_attention: N must be in [1, 2^31)");
    if (T < 1 || T > d.max_len || T > 128) MMT_FAIL("mmt_decode_self_attention: T must be in [1, min(128, pe_trg rows)]");
    if (precision != MMT_PREC_FP32 && precision != MMT_PREC_BF16) MMT_FAIL("bad precision");
    const bool bf16 = precision == MMT_PREC_BF16;
    cudaStream_t s = (cudaStream_t)stream;
    EngineCall call(e, s);
    // the buffers of a one-layer decode wave of N sequences, planned like run_decode's (no cross-attention memory)
    mmt_model_desc d1 = d;
    d1.n_dec_layers = 1;
    Arena ar;
    DecBuffers b;
    MMT_TRY(plan_arena(e, ar, [&]() { plan_decoder(ar, d1, N, 1, 1, T, b, bf16, e->fused_decode_rows); }));
    const int pps = (T + PAGE_TOKENS - 1) / PAGE_TOKENS;
    // unwritten cache slots hold NaN: a key read before it was appended poisons the output instead of passing unnoticed
    MMT_CUDA(cudaMemsetAsync(b.kv_pool, 0xff, (size_t)b.pool_pages * 2 * PAGE_TOKENS * D * b.kv_esz, s));
    prof_pre(e, s);
    init_block_table<<<(unsigned)((N * pps + 255) / 256), 256, 0, s>>>(b.block_table, N, pps);
    MMT_TRY(check_launch(e, "init_block_table", s));
    const int64_t n_el = N * D;
    const unsigned blocks = (unsigned)((n_el + 255) / 256);
    for (int t = 0; t < T; ++t) {
        set_i32<<<1, 1, 0, s>>>(b.ctl, t);
        MMT_TRY(check_launch(e, "set_i32", s));
        if (bf16) {
            f32_to_bf16<<<blocks, 256, 0, s>>>(d_x + t * n_el, n_el, b.x16);
            MMT_TRY(check_launch(e, "f32_to_bf16", s));
        } else MMT_CUDA(cudaMemcpyAsync(b.x, d_x + t * n_el, n_el * sizeof(float), cudaMemcpyDeviceToDevice, s));
        MMT_TRY(decode_self_attention_layer(e, e->dec[layer], b, b.kv_pool, pps, N, bf16, false, s));
        if (bf16) {
            bf16_to_f32<<<blocks, 256, 0, s>>>(b.att16, n_el, d_out + t * n_el);
            MMT_TRY(check_launch(e, "bf16_to_f32", s));
        } else MMT_CUDA(cudaMemcpyAsync(d_out + t * n_el, b.att, n_el * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    return 0;
}

int32_t mmt_decode_cross_attention(mmt_engine* e, const mmt_decode_args* a, int32_t layer, const float* d_q, float* d_out, void* stream) {
    if (!e || !a || !d_q || !d_out) MMT_FAIL("null argument");
    const mmt_model_desc& d = e->desc;
    if (layer < 0 || layer >= d.n_dec_layers) MMT_FAIL("mmt_decode_cross_attention: layer out of range");
    if (a->Bm <= 0 || a->n_cand <= 0 || a->S <= 0) MMT_FAIL("mmt_decode_cross_attention: empty batch");
    if ((a->stride_s % 4) || (a->stride_b % 4) || ((uintptr_t)a->d_memory % 16)) MMT_FAIL("mmt_decode_cross_attention: memory must be 16-byte aligned with strides that are multiples of 4 floats");
    if (a->precision != MMT_PREC_FP32 && a->precision != MMT_PREC_BF16) MMT_FAIL("bad precision");
    const int64_t N = (int64_t)a->Bm * a->n_cand;
    if (N > 0x7fffffff) MMT_FAIL("mmt_decode_cross_attention: too many sequences");
    const bool bf16 = a->precision == MMT_PREC_BF16;
    cudaStream_t s = (cudaStream_t)stream;
    EngineCall call(e, s);
    // one wave of all Bm memories, planned like run_decode's (self-attention cache of a single position)
    Arena ar;
    DecBuffers b;
    MMT_TRY(plan_arena(e, ar, [&]() { plan_decoder(ar, d, N, a->Bm, a->S, 1, b, bf16, e->fused_decode_rows); }));
    MMT_TRY(decode_prepare_wave(e, *a, 0, a->Bm, b, bf16, s));
    MMT_CUDA(cudaMemcpyAsync(b.qc, d_q, (size_t)N * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    const int64_t R = (int64_t)a->Bm * a->S;
    MMT_TRY(decode_cross_attention_layer(e, *a, b, b.cross_kv + (size_t)layer * 2 * R * D * b.kv_esz, N, a->Bm, bf16, false, s));
    if (bf16) {
        bf16_to_f32<<<(unsigned)((N * D + 255) / 256), 256, 0, s>>>(b.att16, N * D, d_out);
        return check_launch(e, "bf16_to_f32", s);
    }
    MMT_CUDA(cudaMemcpyAsync(d_out, b.att, (size_t)N * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}

int32_t mmt_decode_layer_tail(mmt_engine* e, int32_t layer, const float* d_x, const float* d_att_self, const float* d_att_cross,
                              int64_t R, int32_t precision, float* d_x1, float* d_qc, float* d_x2, float* d_out, void* stream) {
    if (!e || !d_x || !d_att_self || !d_att_cross || !d_x1 || !d_qc || !d_out) MMT_FAIL("null argument");
    const mmt_model_desc& d = e->desc;
    if (layer < 0 || layer >= d.n_dec_layers) MMT_FAIL("mmt_decode_layer_tail: layer out of range");
    if (R <= 0 || R > 0x7fffffff) MMT_FAIL("mmt_decode_layer_tail: R must be in [1, 2^31)");
    if (precision != MMT_PREC_FP32 && precision != MMT_PREC_BF16) MMT_FAIL("bad precision");
    const bool bf16 = precision == MMT_PREC_BF16;
    cudaStream_t s = (cudaStream_t)stream;
    EngineCall call(e, s);
    // the buffers of a one-layer decode wave of R sequences, planned like run_decode's
    mmt_model_desc d1 = d;
    d1.n_dec_layers = 1;
    Arena ar;
    DecBuffers b;
    MMT_TRY(plan_arena(e, ar, [&]() { plan_decoder(ar, d1, R, 1, 1, 1, b, bf16, e->fused_decode_rows); }));
    const int64_t n_el = R * D;
    const unsigned blocks = (unsigned)((n_el + 255) / 256);
    const size_t bytes = (size_t)n_el * sizeof(float);
    // an attention output enters the step as att16 (bf16 mode) or att (fp32)
    auto load_att = [&](const float* src) -> int {
        if (bf16) {
            f32_to_bf16<<<blocks, 256, 0, s>>>(src, n_el, b.att16);
            return check_launch(e, "f32_to_bf16", s);
        }
        MMT_CUDA(cudaMemcpyAsync(b.att, src, bytes, cudaMemcpyDeviceToDevice, s));
        return 0;
    };
    const DecOps o{e, b, R, false, s};
    const LayerW& w = e->dec[layer];
    MMT_CUDA(cudaMemcpyAsync(b.x, d_x, bytes, cudaMemcpyDeviceToDevice, s));
    MMT_TRY(load_att(d_att_self));
    MMT_TRY(decode_self_tail_layer(o, w, bf16));
    MMT_CUDA(cudaMemcpyAsync(d_x1, b.x, bytes, cudaMemcpyDeviceToDevice, s));
    MMT_CUDA(cudaMemcpyAsync(d_qc, b.qc, bytes, cudaMemcpyDeviceToDevice, s));
    MMT_TRY(load_att(d_att_cross));
    MMT_TRY(decode_cross_tail_layer(o, w, layer, bf16, d_x2));
    MMT_CUDA(cudaMemcpyAsync(d_out, b.x, bytes, cudaMemcpyDeviceToDevice, s));
    return 0;
}

int32_t mmt_encoder_layer(mmt_engine* e, int32_t stack, int32_t layer, const float* d_x, int64_t rows, int32_t B, int32_t S,
                          const float* d_key_bias, const int32_t* d_row_start, const int32_t* d_cnt, const int32_t* d_kidx,
                          const int32_t* d_nk, int32_t kstride, int32_t precision, float* d_qkv, float* d_att, float* d_out,
                          void* stream) {
    if (!e || !d_x || !d_out) MMT_FAIL("null argument");
    const mmt_model_desc& d = e->desc;
    if (stack < 0 || stack > 5) MMT_FAIL("mmt_encoder_layer: stack must be in [0, 5]");
    if (layer < 0 || layer >= d.n_enc_layers) MMT_FAIL("mmt_encoder_layer: layer out of range");
    if (B <= 0 || B > 65535 || S <= 0 || rows <= 0 || rows > 0x7fffffff) MMT_FAIL("mmt_encoder_layer: empty or oversized batch");
    if (precision != MMT_PREC_FP32 && precision != MMT_PREC_BF16) MMT_FAIL("bad precision");
    const bool ragged = d_key_bias == nullptr;
    if (ragged && (!d_row_start || !d_cnt || !d_kidx || !d_nk || kstride <= 0)) MMT_FAIL("mmt_encoder_layer: the ragged layout needs row_start, cnt, kidx, nk and kstride");
    if (!ragged && rows != (int64_t)B * S) MMT_FAIL("mmt_encoder_layer: the dense layout has B * S rows");
    const bool bf16 = precision == MMT_PREC_BF16;
    const int heads = stack == 5 ? d.n_heads_cross : d.n_heads;
    cudaStream_t s = (cudaStream_t)stream;
    EngineCall call(e, s);
    // the ragged encoder sizes its attention CTAs by the actual per-sequence maxima (encode_chunk_compact reads them back
    // from the index kernels); the dense one by S (max_keys = max_rows = 0)
    int max_keys = 0, max_rows = 0;
    if (ragged) {
        std::vector<int32_t> nk(B), cnt(B), rs(B);
        MMT_CUDA(cudaMemcpyAsync(nk.data(), d_nk, B * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        MMT_CUDA(cudaMemcpyAsync(cnt.data(), d_cnt, B * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        MMT_CUDA(cudaMemcpyAsync(rs.data(), d_row_start, B * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        MMT_CUDA(cudaStreamSynchronize(s));
        for (int b = 0; b < B; ++b) {
            if (nk[b] < 1 || nk[b] > kstride || cnt[b] < 1 || cnt[b] > S || nk[b] > cnt[b] || rs[b] < 0 || rs[b] + (int64_t)cnt[b] > rows)
                MMT_FAIL("mmt_encoder_layer: ragged sequence " + std::to_string(b) + " out of range");
            max_keys = std::max(max_keys, (int)nk[b]); max_rows = std::max(max_rows, (int)cnt[b]);
        }
    }
    Arena a;
    float *X, *QKV, *ATT = nullptr, *PART = nullptr, *H = nullptr;
    __nv_bfloat16 *X16 = nullptr, *ATT16 = nullptr;
    int *kidx = nullptr, *nkd = nullptr;
    auto plan = [&]() {
        X = a.get<float>((size_t)rows * D);
        QKV = a.get<float>((size_t)rows * 3 * D);
        if (bf16) { X16 = a.get<__nv_bfloat16>((size_t)rows * D); ATT16 = a.get<__nv_bfloat16>((size_t)rows * D); }
        else { ATT = a.get<float>((size_t)rows * D); PART = a.get<float>((size_t)rows * D); H = a.get<float>((size_t)rows * d.d_ff); }
        if (!ragged) { kidx = a.get<int>((size_t)B * S); nkd = a.get<int>(B); }
    };
    MMT_TRY(plan_arena(e, a, plan));
    MMT_CUDA(cudaMemcpyAsync(X, d_x, (size_t)rows * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    EncGroupRun g;
    memset(&g, 0, sizeof(g));
    g.X = X; g.rows = (int)rows; g.S = S; g.w = &e->enc[stack][layer];
    g.qkv = QKV; g.att = ATT; g.part = PART; g.h = H; g.x16 = X16; g.att16 = ATT16;
    if (ragged) {
        g.kidx = d_kidx; g.nk = d_nk; g.row_start = d_row_start; g.cnt = d_cnt; g.kstride = kstride;
        g.max_keys = max_keys; g.max_rows = max_rows;
    } else {   // key compaction of the dense encoder (encode_chunk)
        g.kbias = d_key_bias; g.kidx = kidx; g.nk = nkd;
        KeyIndexParams p;
        memset(&p, 0, sizeof(p));
        p.g[0].kbias = d_key_bias; p.g[0].kidx = kidx; p.g[0].nk = nkd; p.g[0].S = S; p.B = B;
        prof_pre(e, s);
        build_key_index<<<dim3(B, 1), 32, 0, s>>>(p);
        MMT_TRY(check_launch(e, "build_key_index", s));
    }
    if (bf16) {
        prof_pre(e, s);
        pack_rows_bf16<<<(unsigned)((rows + 7) / 8), 256, 0, s>>>(X, nullptr, D, rows, X16);
        MMT_TRY(check_launch(e, "pack_rows_bf16", s));
        MMT_TRY(encoder_layer_bf16(e, &g, 1, B, heads, d.d_ff, s));
    } else MMT_TRY(encoder_layer_fp32(e, &g, 1, B, heads, d.d_ff, s));
    if (d_qkv) MMT_CUDA(cudaMemcpyAsync(d_qkv, QKV, (size_t)rows * 3 * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (d_att) {
        if (bf16) {
            bf16_to_f32<<<(unsigned)((rows * D + 255) / 256), 256, 0, s>>>(ATT16, rows * D, d_att);
            MMT_TRY(check_launch(e, "bf16_to_f32", s));
        } else MMT_CUDA(cudaMemcpyAsync(d_att, ATT, (size_t)rows * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    }
    MMT_CUDA(cudaMemcpyAsync(d_out, X, (size_t)rows * D * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
}

int64_t mmt_launch_count(const mmt_engine* e) { return e ? e->launches : 0; }

int32_t mmt_profile_enable(mmt_engine* e, int32_t on) {
    if (!e) MMT_FAIL("null engine");
    std::lock_guard<std::mutex> lk(e->mu);
    for (auto& r : e->prof_records) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    e->prof_records.clear();
    e->profiling = on != 0;
    return 0;
}

int32_t mmt_profile_report(mmt_engine* e, char* buf, int64_t buf_len) {
    if (!e || !buf || buf_len < 2) MMT_FAIL("bad profile buffer");
    std::lock_guard<std::mutex> lk(e->mu);
    MMT_CUDA(cudaSetDevice(e->device));
    MMT_CUDA(cudaDeviceSynchronize());
    struct Agg { int64_t n = 0; double ms = 0, work = 0; };
    std::vector<std::pair<std::string, Agg>> agg;
    for (auto& r : e->prof_records) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
        size_t i = 0;
        for (; i < agg.size(); ++i) if (agg[i].first == r.name) break;
        if (i == agg.size()) agg.push_back({r.name, Agg()});
        agg[i].second.n++; agg[i].second.ms += ms; agg[i].second.work += r.work;
    }
    std::string out = "{";
    for (size_t i = 0; i < agg.size(); ++i) {
        char tmp[256];
        snprintf(tmp, sizeof(tmp), "%s\"%s\": {\"launches\": %lld, \"ms\": %.6f, \"flops\": %.6e}", i ? ", " : "",
                 agg[i].first.c_str(), (long long)agg[i].second.n, agg[i].second.ms, agg[i].second.work);
        out += tmp;
    }
    out += "}";
    if ((int64_t)out.size() + 1 > buf_len) MMT_FAIL("profile buffer too small");
    memcpy(buf, out.c_str(), out.size() + 1);
    return 0;
}

}  // extern "C"
