// fp32 SIMT kernels of the MMT path ("check mode": every contraction is an fp32
// FMA chain so greedy ids reproduce the reference's fp32 PyTorch path), plus the
// kernels that are HBM/latency-bound in every precision mode (embedders, KV-cached
// attention, sampler).
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace mmt {

// ===========================================================================
// GEMM  C[M,N] = act(A[M,K] . W[N,K]^T + bias)     (both operands K-contiguous)
// ===========================================================================
constexpr int GEMM_MAX_GROUPS = 6;

struct GemmGroup {
    const float* A;            // [M, lda]
    const int64_t* a_row_off;  // optional gather: row r of A starts at A + a_row_off[r]
    const float* W;            // [N, K]
    const float* bias;         // [N] or nullptr
    float* C;                  // output
    const int* M_dev;          // optional device-side row count (<= M)
    int64_t lda;
    int M;
};

enum { GEMM_OUT_ROWMAJOR = 0, GEMM_OUT_HEADMAJOR = 1 };

struct GemmParams {
    GemmGroup g[GEMM_MAX_GROUPS];
    int N, K;
    int splits;            // split-K factor; >1 => raw partial sums, no bias/act
    int64_t part_stride;   // floats between consecutive split partials
    int64_t ldc;
    int act;               // 0 none, 1 relu
    int out_mode;          // GEMM_OUT_*
    int hm_heads, hm_dh;   // cross K/V layout, one block per spectrum: r = b*hm_rows + j ->
    int64_t hm_rows;       //   C[(((b*2 + c/D)*heads + (c%D)/dh) * hm_rows + j) * dh + c%dh]
};

template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN))
gemm_nt_f32(const __grid_constant__ GemmParams p) {
    constexpr int BK = 16;
    constexpr int NT = (BM / TM) * (BN / TN);
    constexpr int RV = TM < 4 ? TM : 4;   // rows of a thread come in groups of RV
    constexpr int CV = TN < 4 ? TN : 4;
    constexpr int RG = TM / RV, CG = TN / CV;
    constexpr int LDA_S = BM + 4, LDW_S = BN + 4;
    __shared__ __align__(16) float As[2][BK][LDA_S];
    __shared__ __align__(16) float Ws[2][BK][LDW_S];

    const int grp = blockIdx.z / p.splits, split = blockIdx.z % p.splits;
    const GemmGroup& g = p.g[grp];
    const int M = g.M_dev ? min(*g.M_dev, g.M) : g.M;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    if (m0 >= M) return;
    const int N = p.N, K = p.K;
    int kchunk = ((K / p.splits + BK - 1) / BK) * BK;
    const int kb = split * kchunk;
    const int ke = min(K, kb + kchunk);

    const int tid = threadIdx.x;
    const int tx = tid % (BN / TN), ty = tid / (BN / TN);

    constexpr int A_LD = (BM * 4 + NT - 1) / NT;   // float4 loads per thread for the A tile
    constexpr int W_LD = (BN * 4 + NT - 1) / NT;
    float4 ra[A_LD], rw[W_LD];

    auto load_tiles = [&](int k0) {
#pragma unroll
        for (int i = 0; i < A_LD; ++i) {
            int idx = tid + i * NT;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (idx < BM * 4) {
                int row = idx >> 2, kq = idx & 3;
                int r = m0 + row, k = k0 + kq * 4;
                if (r < M && k < ke) {
                    const float* src = g.a_row_off ? (g.A + g.a_row_off[r]) : (g.A + (int64_t)r * g.lda);
                    if (k + 3 < ke) v = *reinterpret_cast<const float4*>(src + k);
                    else { v.x = src[k]; if (k + 1 < ke) v.y = src[k + 1]; if (k + 2 < ke) v.z = src[k + 2]; }
                }
            }
            ra[i] = v;
        }
#pragma unroll
        for (int i = 0; i < W_LD; ++i) {
            int idx = tid + i * NT;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (idx < BN * 4) {
                int row = idx >> 2, kq = idx & 3;
                int c = n0 + row, k = k0 + kq * 4;
                if (c < N && k < ke) {
                    const float* src = g.W + (int64_t)c * K;
                    if (k + 3 < ke) v = *reinterpret_cast<const float4*>(src + k);
                    else { v.x = src[k]; if (k + 1 < ke) v.y = src[k + 1]; if (k + 2 < ke) v.z = src[k + 2]; }
                }
            }
            rw[i] = v;
        }
    };
    auto store_tiles = [&](int buf) {
#pragma unroll
        for (int i = 0; i < A_LD; ++i) {
            int idx = tid + i * NT;
            if (idx < BM * 4) {
                int row = idx >> 2, kq = (idx & 3) * 4;
                As[buf][kq + 0][row] = ra[i].x; As[buf][kq + 1][row] = ra[i].y;
                As[buf][kq + 2][row] = ra[i].z; As[buf][kq + 3][row] = ra[i].w;
            }
        }
#pragma unroll
        for (int i = 0; i < W_LD; ++i) {
            int idx = tid + i * NT;
            if (idx < BN * 4) {
                int row = idx >> 2, kq = (idx & 3) * 4;
                Ws[buf][kq + 0][row] = rw[i].x; Ws[buf][kq + 1][row] = rw[i].y;
                Ws[buf][kq + 2][row] = rw[i].z; Ws[buf][kq + 3][row] = rw[i].w;
            }
        }
    };

    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    int buf = 0;
    if (kb < ke) {
        load_tiles(kb);
        store_tiles(0);
    }
    __syncthreads();
    for (int k0 = kb; k0 < ke; k0 += BK) {
        const bool more = (k0 + BK) < ke;
        if (more) load_tiles(k0 + BK);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[TM], w[TN];
#pragma unroll
            for (int gi = 0; gi < RG; ++gi)
#pragma unroll
                for (int i = 0; i < RV; ++i) a[gi * RV + i] = As[buf][kk][gi * (BM / RG) + ty * RV + i];
#pragma unroll
            for (int gj = 0; gj < CG; ++gj)
#pragma unroll
                for (int j = 0; j < CV; ++j) w[gj * CV + j] = Ws[buf][kk][gj * (BN / CG) + tx * CV + j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        if (more) {
            store_tiles(buf ^ 1);
            __syncthreads();
            buf ^= 1;
        }
    }

    // epilogue
    float* Cbase = g.C + (p.splits > 1 ? (int64_t)split * p.part_stride : 0);
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        int r = m0 + (i / RV) * (BM / RG) + ty * RV + (i % RV);
        if (r >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            int c = n0 + (j / CV) * (BN / CG) + tx * CV + (j % CV);
            if (c >= N) continue;
            float v = acc[i][j];
            if (p.splits == 1) {
                if (g.bias) v += g.bias[c];
                if (p.act == 1) v = fmaxf(v, 0.f);
            }
            if (p.out_mode == GEMM_OUT_ROWMAJOR) {
                Cbase[(int64_t)r * p.ldc + c] = v;
            } else {
                int kv = c / D, cc = c % D;
                int h = cc / p.hm_dh, d = cc % p.hm_dh;
                const int bb = r / (int)p.hm_rows, jj = r - bb * (int)p.hm_rows;
                Cbase[((((int64_t)bb * 2 + kv) * p.hm_heads + h) * p.hm_rows + jj) * p.hm_dh + d] = v;
            }
        }
    }
}

// ===========================================================================
// out[map(r)] = LayerNorm(res[r] + bias + sum_s part[s][r]) * gamma + beta      (D = 128)
// one warp per row; map(r) = (r / S_in)*stride_b + (r % S_in)*stride_s + off (in rows)
// ===========================================================================
struct LnGroup {
    const float* part;   // [splits][M][D]
    const float* bias;   // [D]
    const float* res;    // [M][D]
    const float* gamma; const float* beta;
    float* out;
    __nv_bfloat16* out_bf16;   // optional bf16 copy, same row map
    const int* M_dev;
    int M;
    int S_in; int64_t stride_b, stride_s, off;
    const int* out_rows;       // optional explicit output row per input row (ragged encoder), overrides the affine map
};
struct LnParams { LnGroup g[GEMM_MAX_GROUPS]; int splits; int64_t part_stride; float eps; };

__global__ void __launch_bounds__(256) bias_res_layernorm(const __grid_constant__ LnParams p) {
    const LnGroup& g = p.g[blockIdx.y];
    const int M = g.M_dev ? min(*g.M_dev, g.M) : g.M;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int r = blockIdx.x * 8 + warp;
    if (r >= M) return;
    const int c = lane * 4;
    float4 v = *reinterpret_cast<const float4*>(g.part + (int64_t)r * D + c);
    for (int s = 1; s < p.splits; ++s) {
        float4 q = *reinterpret_cast<const float4*>(g.part + (int64_t)s * p.part_stride + (int64_t)r * D + c);
        v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    }
    if (g.bias) {
        float4 b = *reinterpret_cast<const float4*>(g.bias + c);
        v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
    }
    if (g.res) {
        float4 q = *reinterpret_cast<const float4*>(g.res + (int64_t)r * D + c);
        v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    }
    float mean = warp_sum(v.x + v.y + v.z + v.w) * (1.0f / D);
    float dx = v.x - mean, dy = v.y - mean, dz = v.z - mean, dw = v.w - mean;
    float var = warp_sum(dx * dx + dy * dy + dz * dz + dw * dw) * (1.0f / D);
    float rstd = rsqrtf(var + p.eps);
    float4 ga = *reinterpret_cast<const float4*>(g.gamma + c);
    float4 be = *reinterpret_cast<const float4*>(g.beta + c);
    float4 o = make_float4(dx * rstd * ga.x + be.x, dy * rstd * ga.y + be.y, dz * rstd * ga.z + be.z, dw * rstd * ga.w + be.w);
    int64_t orow = g.out_rows ? (int64_t)g.out_rows[r] : (int64_t)(r / g.S_in) * g.stride_b + (int64_t)(r % g.S_in) * g.stride_s + g.off;
    *reinterpret_cast<float4*>(g.out + orow * D + c) = o;
    if (g.out_bf16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
        uint2 pk = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        *reinterpret_cast<uint2*>(g.out_bf16 + orow * D + c) = pk;
    }
}

// ===========================================================================
// Encoder input assembly: per-modality sequences [X tokens | MF | MS | MW]
// (reference models_MMT_v15_4.py:733-792 embedders + :549-731 concatenation)
// ===========================================================================
struct EmbedGroup {
    int present;             // 0 => blank modality (zeros + float-ones / bool-false mask)
    int kind;                // 0: 2-col peaks, 1: 1-col peaks (13C), 2: IR (pre-projected row)
    const float* src;        // (B,64,2) | (B,64) | ir_emb (B,D)
    const float* mask;       // (B,64) non-zero = pad; unused for IR
    const float* W;          // (D,2) | (D,1)
    const float* b;          // (D)
    float* X;                // out [B*S_m][D] (modality-encoder input), nullptr when blank
    float* kbias;            // out [B][S_m]  0 / -inf  (modality encoder key bias), nullptr when blank
    int S_m;                 // sequence length of this modality (or blank length)
    int n_x;                 // leading spectrum tokens (64 or 1)
    int off;                 // row offset inside the concatenated memory
    int blank_is_ir;         // blank IR gets a bool False mask (bias 0), others float ones (+1)
    // ragged encoder (kernels_compact.cuh): X row of token (b, s) is row_start[b] + d2c[b][s]; kbias is not written
    const int* d2c; const int* row_start;
};
struct EmbedParams {
    EmbedGroup g[5];
    const int64_t* src_MF; const uint8_t* mask_MF; const float* E_MF; int mf_vocab;
    const int64_t* src_MS; const uint8_t* mask_MS; const float* E_MS; int ms_vocab;
    const float* trg_MW; const float* W_MW; const float* b_MW;
    int has_MF, has_MS, has_MW;
    int B, S_total, P;       // P = pad_points (64); B = spectra in this chunk
    int B_total, b0;         // embedding_src is (S_total, B_total, D); this chunk starts at column b0
    int float_mask;          // concatenated mask promoted to float (pads add +1.0 instead of -inf)
    float* cross_X;          // [B][S_total][D]: only blank rows are written here (zeros)
    float* key_bias;         // out (B,S_total)
    uint8_t* pad_mask;       // out (B,S_total)
    float* embedding_src;    // optional out (S_total,B,D)
};

__global__ void __launch_bounds__(128) embed_tokens(const __grid_constant__ EmbedParams p) {
    const EmbedGroup& g = p.g[blockIdx.y];
    const int b = blockIdx.x, d = threadIdx.x;
    const int B = p.B_total;
    const int bo = p.b0 + b;
    if (!g.present) {
        for (int s = 0; s < g.S_m; ++s) {
            int srow = g.off + s;
            p.cross_X[((int64_t)b * p.S_total + srow) * D + d] = 0.f;
            if (p.embedding_src) p.embedding_src[((int64_t)srow * B + bo) * D + d] = 0.f;
            if (d == 0) {
                p.key_bias[(int64_t)b * p.S_total + srow] = g.blank_is_ir ? 0.f : 1.f;
                p.pad_mask[(int64_t)b * p.S_total + srow] = g.blank_is_ir ? 0 : 1;
            }
        }
        return;
    }
    float w0 = 0.f, w1 = 0.f, bb = 0.f;
    if (g.kind == 0) { w0 = g.W[d * 2]; w1 = g.W[d * 2 + 1]; bb = g.b[d]; }
    else if (g.kind == 1) { w0 = g.W[d]; bb = g.b[d]; }
    const float wmw = p.has_MW ? p.W_MW[d] : 0.f, bmw = p.has_MW ? p.b_MW[d] : 0.f;
    for (int s = 0; s < g.S_m; ++s) {
        float v;
        bool pad;
        int t = s;
        if (t < g.n_x) {
            if (g.kind == 0) {
                const float* x = g.src + ((int64_t)b * p.P + t) * 2;
                v = fmaf(x[1], w1, fmaf(x[0], w0, bb));       // nn.Linear: x0*w0 + x1*w1 + b (order immaterial to 1 ulp)
                pad = g.mask[(int64_t)b * p.P + t] != 0.f;
            } else if (g.kind == 1) {
                v = fmaf(g.src[(int64_t)b * p.P + t], w0, bb);
                pad = g.mask[(int64_t)b * p.P + t] != 0.f;
            } else {
                v = g.src[(int64_t)b * D + d];                 // IR: already relu(W x + b)
                pad = false;
            }
        } else {
            t -= g.n_x;
            if (p.has_MF && t < p.P) {
                int64_t id = p.src_MF[(int64_t)b * p.P + t];
                v = (id >= 0 && id < p.mf_vocab) ? p.E_MF[id * D + d] : 0.f;
                pad = p.mask_MF[(int64_t)b * p.P + t] != 0;
            } else {
                if (p.has_MF) t -= p.P;
                if (p.has_MS && t < p.P) {
                    int64_t id = p.src_MS[(int64_t)b * p.P + t];
                    v = (id >= 0 && id < p.ms_vocab) ? p.E_MS[id * D + d] : 0.f;
                    pad = p.mask_MS[(int64_t)b * p.P + t] != 0;
                } else {
                    v = fmaf(p.trg_MW[b], wmw, bmw);
                    pad = false;
                }
            }
        }
        v = fmaxf(v, 0.f);
        if (g.d2c) g.X[((int64_t)g.row_start[b] + g.d2c[(int64_t)b * CP_SMAX + s]) * D + d] = v;   // padded tokens of a segment share one row (same value)
        else g.X[((int64_t)b * g.S_m + s) * D + d] = v;
        int srow = g.off + s;
        if (p.embedding_src) p.embedding_src[((int64_t)srow * B + bo) * D + d] = v;
        if (d == 0) {
            if (g.kbias) g.kbias[(int64_t)b * g.S_m + s] = pad ? MMT_NEG_INF : 0.f;
            p.key_bias[(int64_t)b * p.S_total + srow] = p.float_mask ? (pad ? 1.f : 0.f) : (pad ? MMT_NEG_INF : 0.f);
            p.pad_mask[(int64_t)b * p.S_total + srow] = pad ? 1 : 0;
        }
    }
}

// ===========================================================================
// Key compaction: indices of keys whose additive bias is not -inf.
// ===========================================================================
struct KeyIndexGroup { const float* kbias; int* kidx; int* nk; int S; };
struct KeyIndexParams { KeyIndexGroup g[GEMM_MAX_GROUPS]; int B; };

__global__ void __launch_bounds__(32) build_key_index(const __grid_constant__ KeyIndexParams p) {
    const KeyIndexGroup& g = p.g[blockIdx.y];
    const int b = blockIdx.x, lane = threadIdx.x;
    int count = 0;
    for (int base = 0; base < g.S; base += 32) {
        int j = base + lane;
        bool valid = j < g.S && g.kbias[(int64_t)b * g.S + j] != MMT_NEG_INF;
        unsigned m = __ballot_sync(0xffffffffu, valid);
        if (valid) g.kidx[(int64_t)b * g.S + count + __popc(m & ((1u << lane) - 1))] = j;
        count += __popc(m);
    }
    if (lane == 0) g.nk[b] = count;
}

// ===========================================================================
// Encoder self-attention, one CTA per (head, sequence, modality); K/V of the
// un-masked keys staged in shared memory; each thread owns query rows.
// ===========================================================================
struct AttnGroup {
    const float* qkv;    // [B*S][3*D]
    const float* kbias;  // [B][S] additive bias per ORIGINAL key index
    const int* kidx;     // [B][S] compacted key indices
    const int* nk;       // [B]
    float* out;          // [B*S][D] fp32 (or nullptr)
    __nv_bfloat16* out16;  // [B*S][D] bf16 operand copy for the tensor-core out-projection (or nullptr)
    int S;
    // ragged encoder: sequence b owns rows [row_start[b], row_start[b] + cnt[b]); kidx rows are kstride apart;
    // every listed key is attendable with bias 0 (kbias == nullptr)
    const int* row_start; const int* cnt; int kstride;
    int smax;              // rows of the K / V staging areas in shared memory (>= keys of any sequence in the launch)
};
struct AttnParams { AttnGroup g[GEMM_MAX_GROUPS]; float scale; };

template <int DH>
__global__ void __launch_bounds__(256) attn_encoder_f32(const __grid_constant__ AttnParams p) {
    extern __shared__ __align__(16) float smem[];
    const AttnGroup& g = p.g[blockIdx.z];
    const int h = blockIdx.x, b = blockIdx.y;
    const int S = g.cnt ? g.cnt[b] : g.S;            // query rows of this sequence
    const int Smax = g.smax;                         // keys the staging area holds (host sizes smem for it)
    const int kstride = g.cnt ? g.kstride : g.S;
    const int64_t row0 = g.row_start ? (int64_t)g.row_start[b] : (int64_t)b * g.S;
    const int nk = g.nk[b];
    float* Ks = smem;                    // [Smax][DH]
    float* Vs = Ks + (size_t)Smax * DH;  // [Smax][DH]
    float* bs = Vs + (size_t)Smax * DH;  // [Smax]
    const float* base = g.qkv + row0 * (3 * D);
    constexpr int V4 = DH / 4;
    // keys [k0, k0 + n) -> shared memory
    auto stage = [&](int k0, int n) {
        for (int i = threadIdx.x; i < n * V4; i += blockDim.x) {
            int jj = i / V4, q4 = i % V4;
            int j = g.kidx[(int64_t)b * kstride + k0 + jj];
            const float* row = base + (int64_t)j * (3 * D) + h * DH + q4 * 4;
            *reinterpret_cast<float4*>(Ks + jj * DH + q4 * 4) = *reinterpret_cast<const float4*>(row + D);
            *reinterpret_cast<float4*>(Vs + jj * DH + q4 * 4) = *reinterpret_cast<const float4*>(row + 2 * D);
            if (q4 == 0) bs[jj] = g.kbias ? g.kbias[(int64_t)b * g.S + j] : 0.f;
        }
    };
    // The usual case stages every key once.  A sequence with more keys than the staging area holds (MS modes with
    // every token valid: up to 902 keys x 260 B > 227 KB) walks them in chunks, re-staged per round of query rows.
    const bool single = nk <= Smax;
    if (single) { stage(0, nk); __syncthreads(); }
    for (int i0 = 0; i0 < S; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool active = i < S;
        float q[DH], acc[DH];
        const float* qrow = base + (int64_t)(active ? i : 0) * (3 * D) + h * DH;
#pragma unroll
        for (int d4 = 0; d4 < V4; ++d4) {
            float4 t = *reinterpret_cast<const float4*>(qrow + d4 * 4);
            q[d4 * 4] = t.x * p.scale; q[d4 * 4 + 1] = t.y * p.scale; q[d4 * 4 + 2] = t.z * p.scale; q[d4 * 4 + 3] = t.w * p.scale;
        }
#pragma unroll
        for (int d = 0; d < DH; ++d) acc[d] = 0.f;
        float m = MMT_NEG_INF, l = 0.f;
        for (int k0 = 0; k0 < nk; k0 += Smax) {
            const int n = min(Smax, nk - k0);
            if (!single) { __syncthreads(); stage(k0, n); __syncthreads(); }
            if (!active) continue;
            for (int j = 0; j < n; ++j) {
                float s = bs[j];
#pragma unroll
                for (int d4 = 0; d4 < V4; ++d4) {
                    float4 k = *reinterpret_cast<const float4*>(Ks + j * DH + d4 * 4);
                    s = fmaf(q[d4 * 4], k.x, s); s = fmaf(q[d4 * 4 + 1], k.y, s);
                    s = fmaf(q[d4 * 4 + 2], k.z, s); s = fmaf(q[d4 * 4 + 3], k.w, s);
                }
                if (s > m) {
                    float corr = expf(m - s);   // m = -inf on the first key -> 0
                    l *= corr;
#pragma unroll
                    for (int d = 0; d < DH; ++d) acc[d] *= corr;
                    m = s;
                }
                float e = expf(s - m);
                l += e;
#pragma unroll
                for (int d4 = 0; d4 < V4; ++d4) {
                    float4 v = *reinterpret_cast<const float4*>(Vs + j * DH + d4 * 4);
                    acc[d4 * 4] = fmaf(e, v.x, acc[d4 * 4]); acc[d4 * 4 + 1] = fmaf(e, v.y, acc[d4 * 4 + 1]);
                    acc[d4 * 4 + 2] = fmaf(e, v.z, acc[d4 * 4 + 2]); acc[d4 * 4 + 3] = fmaf(e, v.w, acc[d4 * 4 + 3]);
                }
            }
        }
        if (!active) continue;
        float inv = 1.0f / l;
        if (g.out) {
            float* orow = g.out + (row0 + i) * D + h * DH;
#pragma unroll
            for (int d4 = 0; d4 < V4; ++d4)
                *reinterpret_cast<float4*>(orow + d4 * 4) =
                    make_float4(acc[d4 * 4] * inv, acc[d4 * 4 + 1] * inv, acc[d4 * 4 + 2] * inv, acc[d4 * 4 + 3] * inv);
        }
        if (g.out16) {
            __nv_bfloat16* orow = g.out16 + (row0 + i) * D + h * DH;
#pragma unroll
            for (int d4 = 0; d4 < V4; ++d4) {
                __nv_bfloat162 lo = __floats2bfloat162_rn(acc[d4 * 4] * inv, acc[d4 * 4 + 1] * inv);
                __nv_bfloat162 hi = __floats2bfloat162_rn(acc[d4 * 4 + 2] * inv, acc[d4 * 4 + 3] * inv);
                *reinterpret_cast<uint2*>(orow + d4 * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Tensor-core variant for the 32-wide heads of encoder_cross (bf16 mode): flash-style attention of one
// (head, sequence) per CTA on mma.sync m16n8k16 (bf16 in, fp32 accumulate).  The operands stay at fp32
// accuracy through two-term bf16 splits -- s = qh.kh + qh.kl + ql.kh, o += ph.vh + ph.vl + pl.vh (the dropped
// lo.lo terms are 2^-18 relative) -- so the kernel changes the speed of the attention, not the numerics of the
// mode.  K and V are staged row-major [key][32] (64-byte rows, 16-byte chunks XOR-swizzled with (key >> 1) & 3:
// conflict-free for ldmatrix) as hi / lo bf16 planes; B fragments come from ldmatrix (K) / ldmatrix.trans (V).  One warp per 16 query rows, keys in
// blocks of 16, online softmax in the log2 domain on the accumulator layout (the score tile's C fragment is
// the P tile's A fragment).
// ---------------------------------------------------------------------------
constexpr int AT_DH = 32;
constexpr int AT_KROW = AT_DH;         // bf16 elements per staged K / V row
// element offset of dims [q4*4, q4*4+4) of key row `key` inside a plane
__device__ __forceinline__ int at_off(int key, int q4) { return key * AT_KROW + ((((q4 >> 1) ^ (key >> 1)) & 3) << 3) + ((q4 & 1) << 2); }

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t saddr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// (x, y) -> packed bf16 hi pair and the packed bf16 pair of the rounding residuals
__device__ __forceinline__ void split_pair(float x, float y, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x, y);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x - __low2float(h), y - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
__host__ __device__ inline int at_keys_padded(int nk) { return (nk + 15) / 16 * 16; }
__host__ __device__ inline size_t at_smem_bytes(int key_bound) {
    const int nkp = at_keys_padded(key_bound);
    return (size_t)4 * nkp * AT_KROW * 2 + (size_t)nkp * 4;
}

__global__ void __launch_bounds__(384, 2) attn_encoder_tc(const __grid_constant__ AttnParams p) {
    extern __shared__ __align__(16) unsigned char at_smem[];
    const AttnGroup& g = p.g[blockIdx.z];
    const int h = blockIdx.x, b = blockIdx.y;
    const int S = g.cnt ? g.cnt[b] : g.S;
    const int kstride = g.cnt ? g.kstride : g.S;
    const int64_t row0 = g.row_start ? (int64_t)g.row_start[b] : (int64_t)b * g.S;
    const int nk = g.nk[b];
    const int nkp_max = at_keys_padded(g.smax);
    const int nkp = at_keys_padded(nk);
    const size_t plane = (size_t)nkp_max * AT_KROW;                  // bf16 elements per plane
    __nv_bfloat16* Kh = reinterpret_cast<__nv_bfloat16*>(at_smem);  // [nkp][AT_KROW] each
    __nv_bfloat16* Kl = Kh + plane;
    __nv_bfloat16* Vh = Kl + plane;
    __nv_bfloat16* Vl = Vh + plane;
    float* bs = reinterpret_cast<float*>(Vl + plane);               // [nkp] key bias * log2(e)
    const float* base = g.qkv + row0 * (3 * D);
    constexpr float LOG2E = 1.4426950408889634f;
    // ---- stage K / V of the attendable keys [k0, k0 + np) as hi / lo bf16 planes; zero the padding keys (>= nk).
    // Four items per thread and pass: the index loads, then the row loads, are all in flight before the first conversion.
    auto stage = [&](int k0, int np) {
    const int total = np * (AT_DH / 4);
    for (int i0 = threadIdx.x; i0 < total; i0 += 4 * blockDim.x) {
        int key[4];
        float4 kk[4], vv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * blockDim.x, jj = i / (AT_DH / 4);
            key[u] = (i < total && k0 + jj < nk) ? g.kidx[(int64_t)b * kstride + k0 + jj] : -1;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * blockDim.x, q4 = i % (AT_DH / 4);
            kk[u] = make_float4(0.f, 0.f, 0.f, 0.f); vv[u] = kk[u];
            if (key[u] >= 0) {
                const float* row = base + (int64_t)key[u] * (3 * D) + h * AT_DH + q4 * 4;
                kk[u] = *reinterpret_cast<const float4*>(row + D);
                vv[u] = *reinterpret_cast<const float4*>(row + 2 * D);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * blockDim.x;
            if (i >= total) break;
            const int jj = i / (AT_DH / 4), q4 = i % (AT_DH / 4);
            if (q4 == 0) bs[jj] = key[u] >= 0 ? (g.kbias ? g.kbias[(int64_t)b * g.S + key[u]] * LOG2E : 0.f) : MMT_NEG_INF;
            uint32_t h0, l0, h1, l1;
            split_pair(kk[u].x, kk[u].y, h0, l0); split_pair(kk[u].z, kk[u].w, h1, l1);
            *reinterpret_cast<uint2*>(Kh + at_off(jj, q4)) = make_uint2(h0, h1);
            *reinterpret_cast<uint2*>(Kl + at_off(jj, q4)) = make_uint2(l0, l1);
            split_pair(vv[u].x, vv[u].y, h0, l0); split_pair(vv[u].z, vv[u].w, h1, l1);
            *reinterpret_cast<uint2*>(Vh + at_off(jj, q4)) = make_uint2(h0, h1);
            *reinterpret_cast<uint2*>(Vl + at_off(jj, q4)) = make_uint2(l0, l1);
        }
    }
    };
    // The usual case stages every key once.  A sequence with more keys than the staging area holds (MS modes with every
    // token valid: 902 keys x 260 B > 227 KB) walks them in chunks, re-staged per round of query-row tiles.
    const bool single = nkp <= nkp_max;
    if (single) { stage(0, nkp); __syncthreads(); }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    // ldmatrix row addresses of this lane (bytes from the plane base, without the key-block offset):
    //   K: matrix lane/8 = dims (lane/8)*8.., row = key (lane%8) of the tile
    //   V (trans): matrix lane/8: keys ((lane/8)&1)*8 + lane%8, dims ((lane/8)>>1)*8..
    // (tile bases are multiples of 8 keys, so the swizzle term depends on lane % 8 only)
    const int sw = (lane & 7) >> 1;
    const uint32_t k_lane_off = (uint32_t)(((lane & 7) * AT_KROW + (((lane >> 3) ^ sw) & 3) * 8) * 2);
    const uint32_t v_row_off = (uint32_t)((((((lane >> 3) & 1) * 8) + (lane & 7)) * AT_KROW) * 2);
    const uint32_t sKh = (uint32_t)__cvta_generic_to_shared(Kh), sKl = (uint32_t)__cvta_generic_to_shared(Kl);
    const uint32_t sVh = (uint32_t)__cvta_generic_to_shared(Vh), sVl = (uint32_t)__cvta_generic_to_shared(Vl);
    const float qscale = p.scale * LOG2E;
    for (int tile0 = 0; tile0 * 16 < S; tile0 += nwarps) {
        const int tile = tile0 + warp;
        const bool active = tile * 16 < S;
        const int r_lo = tile * 16 + gq, r_hi = r_lo + 8;
        // Q fragments (scaled into the log2 domain, split): [kstep][4 regs]
        uint32_t qh[2][4], ql[2][4];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
#pragma unroll
            for (int half = 0; half < 2; ++half) {            // columns ks*16 + 2t (+8)
                const int col = h * AT_DH + ks * 16 + half * 8 + 2 * tq;
                float2 a = make_float2(0.f, 0.f), c = a;
                if (r_lo < S) a = *reinterpret_cast<const float2*>(base + (int64_t)r_lo * (3 * D) + col);
                if (r_hi < S) c = *reinterpret_cast<const float2*>(base + (int64_t)r_hi * (3 * D) + col);
                split_pair(a.x * qscale, a.y * qscale, qh[ks][half * 2], ql[ks][half * 2]);
                split_pair(c.x * qscale, c.y * qscale, qh[ks][half * 2 + 1], ql[ks][half * 2 + 1]);
            }
        float acc[4][4];
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[nt][c] = 0.f;
        float m_lo = MMT_NEG_INF, m_hi = MMT_NEG_INF, l_lo = 0.f, l_hi = 0.f;
        for (int k0 = 0; k0 < nkp; k0 += nkp_max) {
        const int np = min(nkp_max, nkp - k0);
        if (!single) { __syncthreads(); stage(k0, np); __syncthreads(); }
        if (!active) continue;
        for (int kb = 0; kb < np; kb += 16) {
            const uint32_t kb_off = (uint32_t)(kb * AT_KROW * 2);
            // ---- scores of 16 keys: two 16x8 tiles
            float sc[2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(bs + kb + nt * 8 + 2 * tq);
                sc[nt][0] = bb.x; sc[nt][1] = bb.y; sc[nt][2] = bb.x; sc[nt][3] = bb.y;
                uint32_t kh[4], kl[4];          // {b0, b1} of k-step 0, {b0, b1} of k-step 1
                const uint32_t t_off = kb_off + (uint32_t)(nt * 8 * AT_KROW * 2) + k_lane_off;
                ldmatrix_x4(kh, sKh + t_off);
                ldmatrix_x4(kl, sKl + t_off);
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {
                    mma_bf16_16816(sc[nt], qh[ks], kh[ks * 2], kh[ks * 2 + 1]);
                    mma_bf16_16816(sc[nt], qh[ks], kl[ks * 2], kl[ks * 2 + 1]);
                    mma_bf16_16816(sc[nt], ql[ks], kh[ks * 2], kh[ks * 2 + 1]);
                }
            }
            // ---- online softmax over the block (rows g and g+8; a row lives in the 4 lanes of a quad)
            float bm_lo = fmaxf(fmaxf(sc[0][0], sc[0][1]), fmaxf(sc[1][0], sc[1][1]));
            float bm_hi = fmaxf(fmaxf(sc[0][2], sc[0][3]), fmaxf(sc[1][2], sc[1][3]));
            bm_lo = fmaxf(bm_lo, __shfl_xor_sync(0xffffffffu, bm_lo, 1)); bm_lo = fmaxf(bm_lo, __shfl_xor_sync(0xffffffffu, bm_lo, 2));
            bm_hi = fmaxf(bm_hi, __shfl_xor_sync(0xffffffffu, bm_hi, 1)); bm_hi = fmaxf(bm_hi, __shfl_xor_sync(0xffffffffu, bm_hi, 2));
            const float nm_lo = fmaxf(m_lo, bm_lo), nm_hi = fmaxf(m_hi, bm_hi);
            if (__any_sync(0xffffffffu, nm_lo != m_lo || nm_hi != m_hi)) {      // a row maximum moved (else every factor is exactly 1)
                const float corr_lo = ex2_approx(m_lo - nm_lo), corr_hi = ex2_approx(m_hi - nm_hi);     // first block: 2^-inf = 0
                m_lo = nm_lo; m_hi = nm_hi;
                l_lo *= corr_lo; l_hi *= corr_hi;
#pragma unroll
                for (int nt = 0; nt < 4; ++nt) { acc[nt][0] *= corr_lo; acc[nt][1] *= corr_lo; acc[nt][2] *= corr_hi; acc[nt][3] *= corr_hi; }
            }
            uint32_t ph[4], pl[4];      // A fragment of P over the 16 keys: {tile0 row g, tile0 row g+8, tile1 row g, tile1 row g+8}
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float e0 = ex2_approx(sc[nt][0] - m_lo), e1 = ex2_approx(sc[nt][1] - m_lo);
                const float e2 = ex2_approx(sc[nt][2] - m_hi), e3 = ex2_approx(sc[nt][3] - m_hi);
                l_lo += e0 + e1; l_hi += e2 + e3;
                split_pair(e0, e1, ph[nt * 2], pl[nt * 2]);
                split_pair(e2, e3, ph[nt * 2 + 1], pl[nt * 2 + 1]);
            }
            // ---- o += P V  (B fragments by ldmatrix.trans: keys kb + 2t (+8), column d = nt*8 + g)
#pragma unroll
            for (int np2 = 0; np2 < 2; ++np2) {      // pairs of 8-wide output tiles
                uint32_t vh[4], vl[4];            // {b0, b1} of tile 2*np, {b0, b1} of tile 2*np + 1
                const uint32_t t_off = kb_off + v_row_off + (uint32_t)((((np2 * 2 + (lane >> 4)) ^ sw) & 3) * 16);
                ldmatrix_x4_trans(vh, sVh + t_off);
                ldmatrix_x4_trans(vl, sVl + t_off);
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    mma_bf16_16816(acc[np2 * 2 + u], ph, vh[u * 2], vh[u * 2 + 1]);
                    mma_bf16_16816(acc[np2 * 2 + u], ph, vl[u * 2], vl[u * 2 + 1]);
                    mma_bf16_16816(acc[np2 * 2 + u], pl, vh[u * 2], vh[u * 2 + 1]);
                }
            }
        }
        }
        if (!active) continue;
        l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1); l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
        l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1); l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
        const float inv_lo = 1.0f / l_lo, inv_hi = 1.0f / l_hi;
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
            const int col = h * AT_DH + nt * 8 + 2 * tq;
            if (r_lo < S) {
                if (g.out) *reinterpret_cast<float2*>(g.out + (row0 + r_lo) * D + col) = make_float2(acc[nt][0] * inv_lo, acc[nt][1] * inv_lo);
                if (g.out16) *reinterpret_cast<__nv_bfloat162*>(g.out16 + (row0 + r_lo) * D + col) = __floats2bfloat162_rn(acc[nt][0] * inv_lo, acc[nt][1] * inv_lo);
            }
            if (r_hi < S) {
                if (g.out) *reinterpret_cast<float2*>(g.out + (row0 + r_hi) * D + col) = make_float2(acc[nt][2] * inv_hi, acc[nt][3] * inv_hi);
                if (g.out16) *reinterpret_cast<__nv_bfloat162*>(g.out16 + (row0 + r_hi) * D + col) = __floats2bfloat162_rn(acc[nt][2] * inv_hi, acc[nt][3] * inv_hi);
            }
        }
    }
}

// The 8-wide heads of the five modality encoders, same scheme: Q.K^T on m16n8k8, P.V on m16n8k16, every operand a
// two-term bf16 split (three MMAs per product).  K rows are 16 bytes (eight rows = one conflict-free 128-byte line),
// V is staged transposed so that both B fragments are single 32-bit loads.
__device__ __forceinline__ void mma_bf16_1688(float (&c)[4], const uint32_t (&a)[2], uint32_t b0) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(b0));
}
__host__ __device__ inline size_t at8_smem_bytes(int key_bound) {
    const int nkp = at_keys_padded(key_bound);
    return (size_t)2 * nkp * 8 * 2 + (size_t)2 * 8 * (nkp + 8) * 2 + (size_t)nkp * 4;
}
__global__ void __launch_bounds__(128) attn_encoder_tc8(const __grid_constant__ AttnParams p) {
    extern __shared__ __align__(16) unsigned char at_smem[];
    constexpr int DH = 8;
    constexpr float LOG2E = 1.4426950408889634f;
    const AttnGroup& g = p.g[blockIdx.z];
    const int h = blockIdx.x, b = blockIdx.y;
    const int S = g.cnt ? g.cnt[b] : g.S;
    const int kstride = g.cnt ? g.kstride : g.S;
    const int64_t row0 = g.row_start ? (int64_t)g.row_start[b] : (int64_t)b * g.S;
    const int nk = g.nk[b];
    const int nkp_max = at_keys_padded(g.smax), nkp = at_keys_padded(nk);
    const int vstride = nkp_max + 8;
    __nv_bfloat16* Kh = reinterpret_cast<__nv_bfloat16*>(at_smem);      // [nkp][8]
    __nv_bfloat16* Kl = Kh + (size_t)nkp_max * DH;
    __nv_bfloat16* Vh = Kl + (size_t)nkp_max * DH;                      // [8][vstride] (transposed)
    __nv_bfloat16* Vl = Vh + (size_t)DH * vstride;
    float* bs = reinterpret_cast<float*>(Vl + (size_t)DH * vstride);     // [nkp] key bias * log2(e)
    const float* base = g.qkv + row0 * (3 * D);
    for (int i = threadIdx.x; i < nkp * 2; i += blockDim.x) {           // item = (key, half row of four dims)
        const int jj = i >> 1, q4 = i & 1;
        float4 k = make_float4(0.f, 0.f, 0.f, 0.f), v = k;
        if (jj < nk) {
            const int j = g.kidx[(int64_t)b * kstride + jj];
            const float* row = base + (int64_t)j * (3 * D) + h * DH + q4 * 4;
            k = *reinterpret_cast<const float4*>(row + D);
            v = *reinterpret_cast<const float4*>(row + 2 * D);
            if (q4 == 0) bs[jj] = g.kbias ? g.kbias[(int64_t)b * g.S + j] * LOG2E : 0.f;
        } else if (q4 == 0) bs[jj] = MMT_NEG_INF;
        uint32_t h0, l0, h1, l1;
        split_pair(k.x, k.y, h0, l0); split_pair(k.z, k.w, h1, l1);
        *reinterpret_cast<uint2*>(Kh + jj * DH + q4 * 4) = make_uint2(h0, h1);
        *reinterpret_cast<uint2*>(Kl + jj * DH + q4 * 4) = make_uint2(l0, l1);
        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const __nv_bfloat16 vh = __float2bfloat16_rn(vv[c]);
            Vh[(q4 * 4 + c) * vstride + jj] = vh;
            Vl[(q4 * 4 + c) * vstride + jj] = __float2bfloat16_rn(vv[c] - __bfloat162float(vh));
        }
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const float qscale = p.scale * LOG2E;
    for (int tile = warp; tile * 16 < S; tile += nwarps) {
        const int r_lo = tile * 16 + gq, r_hi = r_lo + 8;
        uint32_t qh[2], ql[2];
        {
            const int col = h * DH + 2 * tq;
            float2 a = make_float2(0.f, 0.f), c = a;
            if (r_lo < S) a = *reinterpret_cast<const float2*>(base + (int64_t)r_lo * (3 * D) + col);
            if (r_hi < S) c = *reinterpret_cast<const float2*>(base + (int64_t)r_hi * (3 * D) + col);
            split_pair(a.x * qscale, a.y * qscale, qh[0], ql[0]);
            split_pair(c.x * qscale, c.y * qscale, qh[1], ql[1]);
        }
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        float m_lo = MMT_NEG_INF, m_hi = MMT_NEG_INF, l_lo = 0.f, l_hi = 0.f;
        for (int kb = 0; kb < nkp; kb += 16) {
            float sc[2][4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(bs + kb + nt * 8 + 2 * tq);
                sc[nt][0] = bb.x; sc[nt][1] = bb.y; sc[nt][2] = bb.x; sc[nt][3] = bb.y;
                const uint32_t kh = *reinterpret_cast<const uint32_t*>(Kh + (size_t)(kb + nt * 8 + gq) * DH + 2 * tq);
                const uint32_t kl = *reinterpret_cast<const uint32_t*>(Kl + (size_t)(kb + nt * 8 + gq) * DH + 2 * tq);
                mma_bf16_1688(sc[nt], qh, kh);
                mma_bf16_1688(sc[nt], qh, kl);
                mma_bf16_1688(sc[nt], ql, kh);
            }
            float bm_lo = fmaxf(fmaxf(sc[0][0], sc[0][1]), fmaxf(sc[1][0], sc[1][1]));
            float bm_hi = fmaxf(fmaxf(sc[0][2], sc[0][3]), fmaxf(sc[1][2], sc[1][3]));
            bm_lo = fmaxf(bm_lo, __shfl_xor_sync(0xffffffffu, bm_lo, 1)); bm_lo = fmaxf(bm_lo, __shfl_xor_sync(0xffffffffu, bm_lo, 2));
            bm_hi = fmaxf(bm_hi, __shfl_xor_sync(0xffffffffu, bm_hi, 1)); bm_hi = fmaxf(bm_hi, __shfl_xor_sync(0xffffffffu, bm_hi, 2));
            const float nm_lo = fmaxf(m_lo, bm_lo), nm_hi = fmaxf(m_hi, bm_hi);
            if (__any_sync(0xffffffffu, nm_lo != m_lo || nm_hi != m_hi)) {
                const float corr_lo = ex2_approx(m_lo - nm_lo), corr_hi = ex2_approx(m_hi - nm_hi);
                m_lo = nm_lo; m_hi = nm_hi;
                l_lo *= corr_lo; l_hi *= corr_hi;
                acc[0] *= corr_lo; acc[1] *= corr_lo; acc[2] *= corr_hi; acc[3] *= corr_hi;
            }
            uint32_t ph[4], pl[4];
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const float e0 = ex2_approx(sc[nt][0] - m_lo), e1 = ex2_approx(sc[nt][1] - m_lo);
                const float e2 = ex2_approx(sc[nt][2] - m_hi), e3 = ex2_approx(sc[nt][3] - m_hi);
                l_lo += e0 + e1; l_hi += e2 + e3;
                split_pair(e0, e1, ph[nt * 2], pl[nt * 2]);
                split_pair(e2, e3, ph[nt * 2 + 1], pl[nt * 2 + 1]);
            }
            const uint32_t* vh = reinterpret_cast<const uint32_t*>(Vh + (size_t)gq * vstride + kb + 2 * tq);
            const uint32_t* vl = reinterpret_cast<const uint32_t*>(Vl + (size_t)gq * vstride + kb + 2 * tq);
            const uint32_t vh0 = vh[0], vh1 = vh[4], vl0 = vl[0], vl1 = vl[4];
            mma_bf16_16816(acc, ph, vh0, vh1);
            mma_bf16_16816(acc, ph, vl0, vl1);
            mma_bf16_16816(acc, pl, vh0, vh1);
        }
        l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1); l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
        l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1); l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
        const int col = h * DH + 2 * tq;
        if (r_lo < S) {
            const float o0 = acc[0] / l_lo, o1 = acc[1] / l_lo;
            if (g.out) *reinterpret_cast<float2*>(g.out + (row0 + r_lo) * D + col) = make_float2(o0, o1);
            if (g.out16) *reinterpret_cast<__nv_bfloat162*>(g.out16 + (row0 + r_lo) * D + col) = __floats2bfloat162_rn(o0, o1);
        }
        if (r_hi < S) {
            const float o0 = acc[2] / l_hi, o1 = acc[3] / l_hi;
            if (g.out) *reinterpret_cast<float2*>(g.out + (row0 + r_hi) * D + col) = make_float2(o0, o1);
            if (g.out16) *reinterpret_cast<__nv_bfloat162*>(g.out16 + (row0 + r_hi) * D + col) = __floats2bfloat162_rn(o0, o1);
        }
    }
}

// mean over the S rows of a sequence-first memory (S,B,D) -> (B,D)   (models_MMT_v15_4.py:946)
__global__ void __launch_bounds__(128) mean_over_sequence(const float* mem, int S, int B, float* avg) {
    const int b = blockIdx.x, d = threadIdx.x;
    float s = 0.f;
    for (int i = 0; i < S; ++i) s += mem[((int64_t)i * B + b) * D + d];
    avg[(int64_t)b * D + d] = s / (float)S;
}

// ===========================================================================
// Decoder
// ===========================================================================
// Compact the un-masked memory rows of every memory and record, per packed row,
// where it lives in the caller's (strided, sequence-first) memory tensor.
struct MemIndexParams {
    const float* key_bias;  // (Bm,S)
    int S, Bm;
    int64_t stride_s, stride_b;
    int* nk;                // [Bm]
    int* row_start;         // [Bm]  (= b*S: fixed-stride packing keeps the kernel single-pass)
    int64_t* row_off;       // [Bm*S] float offset of packed row (b*S + jj) in d_memory
    float* kbias_c;         // [Bm*S] bias of packed row
};
__global__ void __launch_bounds__(32) build_memory_index(const MemIndexParams p) {
    const int b = blockIdx.x, lane = threadIdx.x;
    int count = 0;
    for (int base = 0; base < p.S; base += 32) {
        int j = base + lane;
        float bias = j < p.S ? p.key_bias[(int64_t)b * p.S + j] : MMT_NEG_INF;
        bool valid = j < p.S && bias != MMT_NEG_INF;
        unsigned m = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            int pos = b * p.S + count + __popc(m & ((1u << lane) - 1));
            p.row_off[pos] = (int64_t)j * p.stride_s + (int64_t)b * p.stride_b;
            p.kbias_c[pos] = bias;
        }
        count += __popc(m);
    }
    // unused tail rows point at row 0 of this memory so the K/V projection GEMM can run densely
    for (int jj = count + lane; jj < p.S; jj += 32) {
        p.row_off[b * p.S + jj] = (int64_t)b * p.stride_b;
        p.kbias_c[b * p.S + jj] = MMT_NEG_INF;
    }
    if (lane == 0) { p.nk[b] = count; p.row_start[b] = b * p.S; }
}

struct StepCtl {
    int* step;          // device step counter t
    int* done_ctas;     // scratch for the last-CTA-advances-the-step protocol
    int* nonpad;        // [max_len] count of non-<PAD> picks per step
};

// x[n] = E_tok[token_in(t, n)] + E_pos[t]        (validate_generate_MMT_v15_4.py:746-747); orig (compacted wave) or nullptr.
// hist (layer 0 on the position x token table, vocab <= 256): the token also goes to hist[col * hist_ld + t], the history
// decode_self_attention_tm<TmTable> reads -- indexed by the sequence's column, so a compaction moves nothing.
__global__ void __launch_bounds__(128) decode_embed(const int64_t* tokens, int tok_shift, int sos, int64_t N, int64_t ldn,
                                                    const float* E_tok, const float* E_pos, int vocab,
                                                    const int* step, float* x, __nv_bfloat16* x_bf16, const int* orig,
                                                    uint8_t* hist, int hist_ld) {
    pdl_launch_dependents();
    pdl_wait();
    const int t = *step;
    const int64_t n = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (n >= N) return;
    const int lane = threadIdx.x & 31;
    const int64_t col = orig ? orig[n] : n;      // compacted wave (kernels_retire.cuh): row n is sequence orig[n]
    int64_t tok;
    if (tok_shift) tok = (t == 0) ? sos : tokens[(int64_t)(t - 1) * ldn + col];
    else tok = tokens[(int64_t)t * ldn + col];
    if (tok < 0 || tok >= vocab) tok = 0;
    if (hist && lane == 0) hist[col * hist_ld + t] = (uint8_t)tok;
    float4 a = *reinterpret_cast<const float4*>(E_tok + tok * D + lane * 4);
    float4 b = *reinterpret_cast<const float4*>(E_pos + (int64_t)t * D + lane * 4);
    float4 o = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    *reinterpret_cast<float4*>(x + n * D + lane * 4) = o;
    if (x_bf16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
        *reinterpret_cast<uint2*>(x_bf16 + n * D + lane * 4) =
            make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
    }
}

// Causal self-attention of the new position over the paged KV cache; one warp per
// (sequence, head).  Appends this step's K,V to the cache first.
// page layout: [2 (K,V)][H][PAGE_TOKENS][DH] elements of KVT (fp32 check mode / bf16 tensor-core mode).
template <int DH, typename KVT>
__global__ void __launch_bounds__(256) decode_self_attention(const float* qkv, KVT* kv_pool, const int* block_table,
                                                             int pages_per_seq, int64_t N, int H, float scale,
                                                             const int* step, float* out, __nv_bfloat16* out16) {
    static_assert(DH == 8, "8-element key rows");
    typedef KvRow<KVT> KV;
    const int t = *step;
    const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= N * H) return;
    const int lane = threadIdx.x & 31;
    const int64_t n = w / H;
    const int h = (int)(w % H);
    constexpr int PAGE_ELEMS = 2 * PAGE_TOKENS * D;
    const int* bt = block_table + n * pages_per_seq;
    const float* row = qkv + n * (3 * D) + h * DH;
    // append K,V of position t
    if (lane < 2 * DH) {
        int kv = lane / DH, d = lane % DH;
        KVT* page = kv_pool + (int64_t)bt[t / PAGE_TOKENS] * PAGE_ELEMS;
        KV::st(page + ((kv * H + h) * PAGE_TOKENS + (t % PAGE_TOKENS)) * DH + d, row[(1 + kv) * D + d]);
    }
    __syncwarp();
    float q[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) q[d] = row[d] * scale;
    // pass 1: scores (each lane owns keys lane, lane+32, ...)
    constexpr int MAXK = 4;   // max_len 128 / 32
    float s[MAXK];
    float m = MMT_NEG_INF;
#pragma unroll
    for (int i = 0; i < MAXK; ++i) {
        int j = lane + i * 32;
        s[i] = MMT_NEG_INF;
        if (j <= t) {
            const KVT* page = kv_pool + (int64_t)bt[j / PAGE_TOKENS] * PAGE_ELEMS;
            float k[DH];
            KV::unpack(KV::ld(page + ((0 * H + h) * PAGE_TOKENS + (j % PAGE_TOKENS)) * DH), k);
            float a = 0.f;
#pragma unroll
            for (int d = 0; d < DH; ++d) a = fmaf(q[d], k[d], a);
            s[i] = a;
            m = fmaxf(m, a);
        }
    }
    m = warp_max(m);
    float l = 0.f, acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = 0.f;
#pragma unroll
    for (int i = 0; i < MAXK; ++i) {
        int j = lane + i * 32;
        if (j <= t) {
            float e = expf(s[i] - m);
            l += e;
            const KVT* page = kv_pool + (int64_t)bt[j / PAGE_TOKENS] * PAGE_ELEMS;
            float v[DH];
            KV::unpack(KV::ld(page + ((1 * H + h) * PAGE_TOKENS + (j % PAGE_TOKENS)) * DH), v);
#pragma unroll
            for (int d = 0; d < DH; ++d) acc[d] = fmaf(e, v[d], acc[d]);
        }
    }
    l = warp_sum(l);
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = warp_sum(acc[d]);
    if (lane < DH) {
        float v = 0.f;
#pragma unroll
        for (int d = 0; d < DH; ++d) if (lane == d) v = acc[d];
        if (out) out[n * D + h * DH + lane] = v / l;
        if (out16) out16[n * D + h * DH + lane] = __float2bfloat16_rn(v / l);
    }
}

// The same, eight lanes per (sequence, head): a warp serves four heads of a sequence, lane (hq, kl) owns the keys
// j = kl (mod 8) of head hq.  At the positions where most of a 128-token decode lives (t < 64) a warp-per-head mapping
// leaves most lanes without a key and still pays a five-stage reduction of ten values; here the reduction is three
// stages over eight lanes (8-value reduce-scatter: lane kl ends up with output dimension kl, so a warp stores 32
// consecutive outputs) and the wave needs a quarter of the warps.  Online softmax, two keys per lane in flight.
// APPEND = false: K / V of position t are already in the cache (written by the QKV projection's epilogue, kernels_tc.cuh).
template <int DH, typename KVT, bool APPEND = true>
__global__ void __launch_bounds__(256) decode_self_attention_g8(const float* qkv, KVT* kv_pool, const int* block_table,
                                                                int pages_per_seq, int64_t N, int H, float scale,
                                                                const int* step, float* out, __nv_bfloat16* out16) {
    static_assert(DH == 8, "8-element key rows");
    typedef KvRow<KVT> KV;
    pdl_launch_dependents();
    pdl_wait();
    const int t = *step;
    const int HG = H / 4;                                  // head groups per sequence
    const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= N * HG) return;
    const int lane = threadIdx.x & 31, hq = lane >> 3, kl = lane & 7;
    const int64_t n = w / HG;
    const int h = (int)(w % HG) * 4 + hq;
    constexpr int PAGE_ELEMS = 2 * PAGE_TOKENS * D;
    const int* bt = block_table + n * pages_per_seq;
    const float* row = qkv + n * (APPEND ? 3 * D : D) + h * DH;      // APPEND = false: `qkv` is the dense [N][D] query buffer
    if (APPEND) {   // append K,V of position t: lane (hq, kl) writes element kl of its head's K and V rows
        KVT* page = kv_pool + (int64_t)bt[t / PAGE_TOKENS] * PAGE_ELEMS;
        KV::st(page + ((0 * H + h) * PAGE_TOKENS + (t % PAGE_TOKENS)) * DH + kl, row[D + kl]);
        KV::st(page + ((1 * H + h) * PAGE_TOKENS + (t % PAGE_TOKENS)) * DH + kl, row[2 * D + kl]);
        __syncwarp();
    }
    float q[DH], acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) { q[d] = row[d] * scale; acc[d] = 0.f; }
    float m = MMT_NEG_INF, l = 0.f;
    // software pipeline: the K/V rows of the next two keys are in flight while the current two are folded in
    auto row_ptr = [&](int j) { return kv_pool + (int64_t)bt[j / PAGE_TOKENS] * PAGE_ELEMS + (h * PAGE_TOKENS + (j % PAGE_TOKENS)) * DH; };
    typename KV::Raw rk0, rk1, rv0, rv1;
    if (kl <= t) {
        const KVT* p0 = row_ptr(kl);
        const KVT* p1 = row_ptr(kl + 8 <= t ? kl + 8 : kl);
        rk0 = KV::ld(p0); rk1 = KV::ld(p1);
        rv0 = KV::ld(p0 + H * PAGE_TOKENS * DH); rv1 = KV::ld(p1 + H * PAGE_TOKENS * DH);
    }
    for (int j0 = kl; j0 <= t; j0 += 16) {
        const bool has1 = j0 + 8 <= t;
        const typename KV::Raw ck0 = rk0, ck1 = rk1, cv0 = rv0, cv1 = rv1;
        const int jn = j0 + 16;
        if (jn <= t) {
            const KVT* p0 = row_ptr(jn);
            const KVT* p1 = row_ptr(jn + 8 <= t ? jn + 8 : jn);
            rk0 = KV::ld(p0); rk1 = KV::ld(p1);
            rv0 = KV::ld(p0 + H * PAGE_TOKENS * DH); rv1 = KV::ld(p1 + H * PAGE_TOKENS * DH);
        }
        float k0[DH], k1[DH];
        KV::unpack(ck0, k0); KV::unpack(ck1, k1);
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int d = 0; d < DH; ++d) { s0 = fmaf(q[d], k0[d], s0); s1 = fmaf(q[d], k1[d], s1); }
        if (!has1) s1 = MMT_NEG_INF;
        const float mn = fmaxf(m, fmaxf(s0, s1));
        if (mn > m) {
            const float corr = expf(m - mn);
            l *= corr;
#pragma unroll
            for (int d = 0; d < DH; ++d) acc[d] *= corr;
            m = mn;
        }
        const float e0 = expf(s0 - m), e1 = has1 ? expf(s1 - m) : 0.f;
        l += e0 + e1;
        float v0[DH], v1[DH];
        KV::unpack(cv0, v0); KV::unpack(cv1, v1);
#pragma unroll
        for (int d = 0; d < DH; ++d) acc[d] = fmaf(e1, v1[d], fmaf(e0, v0[d], acc[d]));
    }
    // merge the eight per-lane partial softmaxes of a head (lanes without a key carry m = -inf, l = 0)
    float Mx = m;
    Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, 1)); Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, 2)); Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, 4));
    const float corr = (m == MMT_NEG_INF) ? 0.f : expf(m - Mx);
    l *= corr;
    l += __shfl_xor_sync(0xffffffffu, l, 1); l += __shfl_xor_sync(0xffffffffu, l, 2); l += __shfl_xor_sync(0xffffffffu, l, 4);
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] *= corr;
#pragma unroll
    for (int off = 4; off >= 1; off >>= 1) {          // 8-value reduce-scatter over the 8 lanes: lane kl keeps dimension kl
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            const float send = up ? acc[i] : acc[i + off];
            const float keep = up ? acc[i + off] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    const float o = acc[0] / l;
    if (out) out[n * D + h * DH + kl] = o;
    if (out16) out16[n * D + h * DH + kl] = __float2bfloat16_rn(o);
}

// Large bf16 waves: TOKEN-MAJOR pages, [PAGE_TOKENS][2 (K,V)][H][DH] -- the K | V of one token are 512 contiguous bytes.
// With the head-major page every (K|V, head) plane of the OPEN page is a 256-byte run of which (t % 16 + 1) x 16 bytes are
// valid, and the memory system fetches the whole 128-byte lines: ncu read the full 8 KB of the open page at every step
// (1902 MB of DRAM reads against 1670 MB of valid rows at t = 41).  Token-major, the valid tokens of the open page are one
// contiguous prefix, and the QKV projection's epilogue appends a token as two 256-byte row segments instead of 32 scattered
// 16-byte pieces.  Mapping: a warp serves eight heads of a sequence, lane (h8, kl) owns the keys j = kl (mod 4) of head h8:
// one load instruction covers 4 tokens x 128 contiguous bytes.  Online softmax, two keys per lane in flight and two more
// prefetched; the 8 output dimensions are reduce-scattered over the 4 lanes of a head (lane kl keeps dimensions 2 kl,
// 2 kl + 1), so a warp stores 128 consecutive bytes.  K / V of position t are already in the cache (kernels_tc.cuh).
// The row source Src gives, per sequence, the query row of position t and the K | V row of key j (512 bytes: K of every
// head, then V -- the token-major page row): TmPaged (the cache) or TmTable (decoder layer 0).
struct TmPaged {     // query: the QKV projection's dense [N][D] Q output; key j: slot j % 16 of page block_table[n][j / 16]
    const float* qd; const __nv_bfloat16* kv_pool; const int* block_table; int pps;
    struct Seq {
        const float* q; const __nv_bfloat16* pool; const int* bt;
        __device__ __forceinline__ const float* q_row(int) const { return q; }
        __device__ __forceinline__ const __nv_bfloat16* kv_row(int j) const {
            return pool + (int64_t)bt[j / PAGE_TOKENS] * (2 * PAGE_TOKENS * D) + (j % PAGE_TOKENS) * (2 * D);
        }
    };
    __device__ __forceinline__ Seq seq(int64_t n) const { return {qd + n * D, kv_pool, block_table + n * pps}; }
};
// Decoder layer 0: its input at position j is E_tok[tok_j] + E_pos[j], so its Q and K | V rows depend on (j, tok_j) alone.
// qtab [pos][tok][D] fp32 and kvtab [pos][tok][2 D] bf16 hold them for every pair (built once per engine, engine.cu
// ensure_l0_table, by the same projection as the step's); tok_j comes from the sequence's token history (decode_embed),
// row hist_ld * col, col = orig[n] in a compacted wave.  Plain cached loads: rows shared by many sequences (every
// sequence's key 0 is the same <SOS> row) stay in L1.
struct TmTable {
    const float* qtab; const __nv_bfloat16* kvtab; const uint8_t* hist; int hist_ld; int vocab; const int* orig;
    struct Seq {
        const float* qtab; const __nv_bfloat16* kvtab; const uint8_t* hist; int vocab;
        __device__ __forceinline__ const float* q_row(int t) const { return qtab + ((int64_t)t * vocab + hist[t]) * D; }
        __device__ __forceinline__ const __nv_bfloat16* kv_row(int j) const { return kvtab + ((int64_t)j * vocab + hist[j]) * (2 * D); }
    };
    __device__ __forceinline__ Seq seq(int64_t n) const {
        return {qtab, kvtab, hist + (int64_t)(orig ? orig[n] : n) * hist_ld, vocab};
    }
};
template <int DH, class Src>
__global__ void __launch_bounds__(256) decode_self_attention_tm(const Src src, int64_t N, int H, float scale,
                                                                const int* step, __nv_bfloat16* out16) {
    static_assert(DH == 8, "8-element key rows");
    typedef KvRow<__nv_bfloat16> KV;
    pdl_launch_dependents();
    pdl_wait();
    const int t = *step;
    const int HG = H / 8;                                  // head groups per sequence
    const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= N * HG) return;
    const int lane = threadIdx.x & 31, h8 = lane >> 2, kl = lane & 3;
    const int64_t n = w / HG;
    const int h = (int)(w % HG) * 8 + h8;
    const typename Src::Seq sq = src.seq(n);
    const float* row = sq.q_row(t) + h * DH;
    float q[DH], acc[DH];
    {
        const float4 a = *reinterpret_cast<const float4*>(row), b = *reinterpret_cast<const float4*>(row + 4);
        q[0] = a.x * scale; q[1] = a.y * scale; q[2] = a.z * scale; q[3] = a.w * scale;
        q[4] = b.x * scale; q[5] = b.y * scale; q[6] = b.z * scale; q[7] = b.w * scale;
    }
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = 0.f;
    float m = MMT_NEG_INF, l = 0.f;
    auto row_ptr = [&](int j) { return sq.kv_row(j) + h * DH; };
    typename KV::Raw rk0, rk1, rv0, rv1;
    if (kl <= t) {
        const __nv_bfloat16* p0 = row_ptr(kl);
        const __nv_bfloat16* p1 = row_ptr(kl + 4 <= t ? kl + 4 : kl);
        rk0 = KV::ld(p0); rk1 = KV::ld(p1);
        rv0 = KV::ld(p0 + D); rv1 = KV::ld(p1 + D);
    }
    for (int j0 = kl; j0 <= t; j0 += 8) {
        const bool has1 = j0 + 4 <= t;
        const typename KV::Raw ck0 = rk0, ck1 = rk1, cv0 = rv0, cv1 = rv1;
        const int jn = j0 + 8;
        if (jn <= t) {
            const __nv_bfloat16* p0 = row_ptr(jn);
            const __nv_bfloat16* p1 = row_ptr(jn + 4 <= t ? jn + 4 : jn);
            rk0 = KV::ld(p0); rk1 = KV::ld(p1);
            rv0 = KV::ld(p0 + D); rv1 = KV::ld(p1 + D);
        }
        float k0[DH], k1[DH];
        KV::unpack(ck0, k0); KV::unpack(ck1, k1);
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int d = 0; d < DH; ++d) { s0 = fmaf(q[d], k0[d], s0); s1 = fmaf(q[d], k1[d], s1); }
        if (!has1) s1 = MMT_NEG_INF;
        const float mn = fmaxf(m, fmaxf(s0, s1));
        if (mn > m) {
            const float corr = expf(m - mn);
            l *= corr;
#pragma unroll
            for (int d = 0; d < DH; ++d) acc[d] *= corr;
            m = mn;
        }
        const float e0 = expf(s0 - m), e1 = has1 ? expf(s1 - m) : 0.f;
        l += e0 + e1;
        float v0[DH], v1[DH];
        KV::unpack(cv0, v0); KV::unpack(cv1, v1);
#pragma unroll
        for (int d = 0; d < DH; ++d) acc[d] = fmaf(e1, v1[d], fmaf(e0, v0[d], acc[d]));
    }
    // merge the four per-lane partial softmaxes of a head (lanes without a key carry m = -inf, l = 0)
    float Mx = m;
    Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, 1)); Mx = fmaxf(Mx, __shfl_xor_sync(0xffffffffu, Mx, 2));
    const float corr = (m == MMT_NEG_INF) ? 0.f : expf(m - Mx);
    l *= corr;
    l += __shfl_xor_sync(0xffffffffu, l, 1); l += __shfl_xor_sync(0xffffffffu, l, 2);
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] *= corr;
#pragma unroll
    for (int off = 2; off >= 1; off >>= 1) {          // 8-value reduce-scatter over the 4 lanes: lane kl keeps dimensions 2 kl, 2 kl + 1
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < 2 * off; ++i) {
            const float send = up ? acc[i] : acc[i + 2 * off];
            const float keep = up ? acc[i + 2 * off] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    const __nv_bfloat162 o = __floats2bfloat162_rn(acc[0] / l, acc[1] / l);
    *reinterpret_cast<__nv_bfloat162*>(out16 + n * D + h * DH + 2 * kl) = o;
}

// Layer-0 table (TmTable), input rows: row r = t * vocab + tok is bf16(E_tok[tok] + E_pos[t]), decode_embed's arithmetic
__global__ void __launch_bounds__(128) l0_table_rows(const float* E_tok, const float* E_pos, int vocab, int64_t rows, __nv_bfloat16* out) {
    const int64_t r = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (r >= rows) return;
    const int lane = threadIdx.x & 31;
    const int64_t t = r / vocab, tok = r % vocab;
    const float4 a = *reinterpret_cast<const float4*>(E_tok + tok * D + lane * 4);
    const float4 b = *reinterpret_cast<const float4*>(E_pos + t * D + lane * 4);
    const float4 o = make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
    __nv_bfloat162 lo = __floats2bfloat162_rn(o.x, o.y), hi = __floats2bfloat162_rn(o.z, o.w);
    *reinterpret_cast<uint2*>(out + r * D + lane * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
}

// Layer-0 table: the projected rows [rows][Q | K | V] (fp32, bias added) -> qtab [rows][D] fp32 and kvtab [rows][K | V] bf16,
// rounded like the KV-append epilogue (kernels_tc.cuh pack_bf16x4)
__global__ void __launch_bounds__(128) l0_table_split(const float* qkv, int64_t rows, float* qtab, __nv_bfloat16* kvtab) {
    const int64_t r = (int64_t)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (r >= rows) return;
    const int lane = threadIdx.x & 31;
    const float* src = qkv + r * (3 * D);
    *reinterpret_cast<float4*>(qtab + r * D + lane * 4) = *reinterpret_cast<const float4*>(src + lane * 4);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const float4 v = *reinterpret_cast<const float4*>(src + D + c * D + lane * 4);
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        *reinterpret_cast<uint2*>(kvtab + r * (2 * D) + c * D + lane * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
    }
}

// Cross-attention of the new position over the (compacted) projected memory;
// one warp per (sequence, head).  K/V layout: [spectrum][K|V][H][rows_total = rows per spectrum][DH] of KVT.
template <int DH, typename KVT>
__global__ void __launch_bounds__(256) decode_cross_attention(const float* q_in, const KVT* kv, int64_t rows_total,
                                                              const int* nk, const int* row_start, const float* kbias_c,
                                                              int n_cand, int64_t N, int H, float scale, float* out,
                                                              __nv_bfloat16* out16, const int* orig) {
    static_assert(DH == 8, "8-element key rows");
    typedef KvRow<KVT> KV;
    pdl_launch_dependents();
    pdl_wait();
    const int64_t w = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (w >= N * H) return;
    const int lane = threadIdx.x & 31;
    const int64_t n = w / H;
    const int h = (int)(w % H);
    const int64_t b = (orig ? orig[n] : n) / n_cand;      // compacted wave: row n is sequence orig[n]
    const int cnt = nk[b];
    const int64_t r0 = row_start[b];
    // one contiguous K/V block per spectrum: [K|V][H][S][DH], S = rows reserved per spectrum (r0 = b * S)
    const int64_t S = rows_total;
    const KVT* Kh = kv + (((int64_t)b * 2 + 0) * H + h) * S * DH;
    const KVT* Vh = kv + (((int64_t)b * 2 + 1) * H + h) * S * DH;
    const float* bias = kbias_c + r0;
    float q[DH], acc[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) { q[d] = q_in[n * D + h * DH + d] * scale; acc[d] = 0.f; }
    float m = MMT_NEG_INF, l = 0.f;
    for (int j = lane; j < cnt; j += 32) {
        const typename KV::Raw rk = KV::ld(Kh + (int64_t)j * DH), rv = KV::ld(Vh + (int64_t)j * DH);
        float s = bias[j];
        float k[DH];
        KV::unpack(rk, k);
#pragma unroll
        for (int d = 0; d < DH; ++d) s = fmaf(q[d], k[d], s);
        if (s > m) {
            float corr = expf(m - s);
            l *= corr;
#pragma unroll
            for (int d = 0; d < DH; ++d) acc[d] *= corr;
            m = s;
        }
        float e = expf(s - m);
        l += e;
        float v[DH];
        KV::unpack(rv, v);
#pragma unroll
        for (int d = 0; d < DH; ++d) acc[d] = fmaf(e, v[d], acc[d]);
    }
    // merge the 32 per-lane partial softmaxes
    float M = warp_max(m);
    float corr = (m == MMT_NEG_INF) ? 0.f : expf(m - M);
    l = warp_sum(l * corr);
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = warp_sum(acc[d] * corr);
    if (lane < DH) {
        float v = 0.f;
#pragma unroll
        for (int d = 0; d < DH; ++d) if (lane == d) v = acc[d];
        if (out) out[n * D + h * DH + lane] = v / l;
        if (out16) out16[n * D + h * DH + lane] = __float2bfloat16_rn(v / l);
    }
}

// Tensor-core cross-attention for candidate waves (bf16 K/V): the n_cand sequences of a spectrum attend to the SAME
// projected memory (run_batch_gen_val_MMT_v15_4.py:93-158 decodes 128 candidates per spectrum), so per (spectrum, head)
// the scores are a real [n_cand x 8] . [8 x keys] product and the output a [n_cand x keys] . [keys x 8] one.  One CTA
// per (head, spectrum) stages that head's K (row-major) and V (transposed) once; a warp owns 16 candidates: Q.K^T on
// mma.sync m16n8k8, P.V on m16n8k16, online softmax in the log2 domain on the accumulator layout.  Q enters as a
// two-term bf16 split (K and V are bf16 already): the scores equal the SIMT kernel's to fp32 round-off; P is bf16.
__host__ __device__ inline int dx_keys_padded(int nk) { return (nk + 31) / 32 * 32; }      // 32 keys per softmax round
__host__ __device__ inline size_t dx_smem_bytes(int key_bound) {
    const int nkp = dx_keys_padded(key_bound);
    return (size_t)nkp * 8 * 2 + (size_t)8 * (nkp + 8) * 2 + (size_t)nkp * 4;
}
__global__ void __launch_bounds__(256) decode_cross_attention_tc(const float* q_in, const __nv_bfloat16* kv, int64_t rows_total,
                                                                 const int* nk, const int* row_start, const float* kbias_c,
                                                                 int n_cand, int H, float scale, float* out, __nv_bfloat16* out16,
                                                                 const int* col_start, const int* col_count) {
    extern __shared__ __align__(16) unsigned char dx_smem[];
    constexpr int DH = 8;
    constexpr float LOG2E = 1.4426950408889634f;
    pdl_launch_dependents();
    const int h = blockIdx.x;
    const int64_t b = blockIdx.y;
    // compacted wave (kernels_retire.cuh): column b's candidates are rows col_start[b] .. + col_count[b]
    const int nc = col_count ? col_count[b] : n_cand;
    const int64_t row0 = col_count ? (int64_t)col_start[b] : b * n_cand;
    if (nc == 0) return;
    const int cnt = nk[b];
    const int64_t r0 = row_start[b];
    const int nkp_max = dx_keys_padded((int)rows_total), nkp = dx_keys_padded(cnt);
    const int vstride = nkp_max + 8;
    __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(dx_smem);           // [nkp][8]
    __nv_bfloat16* Vt = Ks + (size_t)nkp_max * DH;                           // [8][vstride]
    float* bs = reinterpret_cast<float*>(Vt + (size_t)DH * vstride);          // [nkp] bias * log2(e)
    const __nv_bfloat16* Kh = kv + (((int64_t)b * 2 + 0) * H + h) * rows_total * DH;
    const __nv_bfloat16* Vh = kv + (((int64_t)b * 2 + 1) * H + h) * rows_total * DH;
    for (int j = threadIdx.x; j < nkp; j += blockDim.x) {
        uint4 k = make_uint4(0u, 0u, 0u, 0u), v = k;
        float bias = MMT_NEG_INF;
        if (j < cnt) {
            k = *reinterpret_cast<const uint4*>(Kh + (int64_t)j * DH);
            v = *reinterpret_cast<const uint4*>(Vh + (int64_t)j * DH);
            bias = kbias_c[r0 + j] * LOG2E;
        }
        *reinterpret_cast<uint4*>(Ks + (size_t)j * DH) = k;
        const uint32_t vw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            Vt[(2 * c) * vstride + j] = __ushort_as_bfloat16((unsigned short)(vw[c] & 0xffffu));
            Vt[(2 * c + 1) * vstride + j] = __ushort_as_bfloat16((unsigned short)(vw[c] >> 16));
        }
        bs[j] = bias;
    }
    __syncthreads();
    pdl_wait();     // everything above reads decode-loop constants (projected memory, key counts, biases); the queries are the predecessor's
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int gq = lane >> 2, tq = lane & 3;
    const float qscale = scale * LOG2E;
    for (int tile = warp; tile * 16 < nc; tile += nwarps) {
        const int c_lo = tile * 16 + gq, c_hi = c_lo + 8;
        const int64_t n_lo = row0 + c_lo, n_hi = row0 + c_hi;
        uint32_t qh[2], ql[2];
        {
            float2 a = make_float2(0.f, 0.f), c = a;
            if (c_lo < nc) a = *reinterpret_cast<const float2*>(q_in + n_lo * D + h * DH + 2 * tq);
            if (c_hi < nc) c = *reinterpret_cast<const float2*>(q_in + n_hi * D + h * DH + 2 * tq);
            split_pair(a.x * qscale, a.y * qscale, qh[0], ql[0]);
            split_pair(c.x * qscale, c.y * qscale, qh[1], ql[1]);
        }
        const uint32_t qa[4] = {qh[0], qh[1], ql[0], ql[1]};      // m16n8k16 A fragment: columns 0-7 = Q_hi, 8-15 = Q_lo
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        float m_lo = MMT_NEG_INF, m_hi = MMT_NEG_INF, l_lo = 0.f, l_hi = 0.f;
        // 32 keys per round: four score tiles first, ONE running-max update for all of them, then the exponentials and two P.V
        // MMAs -- half the max / shuffle / rescale bookkeeping per key of a 16-key round and twice the independent work in flight
        for (int kb = 0; kb < nkp; kb += 32) {
            float sc[4][4];
#pragma unroll
            for (int nt = 0; nt < 4; ++nt) {
                const float2 bb = *reinterpret_cast<const float2*>(bs + kb + nt * 8 + 2 * tq);
                sc[nt][0] = bb.x; sc[nt][1] = bb.y; sc[nt][2] = bb.x; sc[nt][3] = bb.y;
                const uint32_t kf = *reinterpret_cast<const uint32_t*>(Ks + (size_t)(kb + nt * 8 + gq) * DH + 2 * tq);
                mma_bf16_16816(sc[nt], qa, kf, kf);        // [Q_hi | Q_lo] (k = 16) . [K ; K]: both terms of Q in one instruction
            }
            float bm_lo = fmaxf(fmaxf(fmaxf(sc[0][0], sc[0][1]), fmaxf(sc[1][0], sc[1][1])), fmaxf(fmaxf(sc[2][0], sc[2][1]), fmaxf(sc[3][0], sc[3][1])));
            float bm_hi = fmaxf(fmaxf(fmaxf(sc[0][2], sc[0][3]), fmaxf(sc[1][2], sc[1][3])), fmaxf(fmaxf(sc[2][2], sc[2][3]), fmaxf(sc[3][2], sc[3][3])));
            bm_lo = fmaxf(bm_lo, __shfl_xor_sync(0xffffffffu, bm_lo, 1)); bm_lo = fmaxf(bm_lo, __shfl_xor_sync(0xffffffffu, bm_lo, 2));
            bm_hi = fmaxf(bm_hi, __shfl_xor_sync(0xffffffffu, bm_hi, 1)); bm_hi = fmaxf(bm_hi, __shfl_xor_sync(0xffffffffu, bm_hi, 2));
            const float nm_lo = fmaxf(m_lo, bm_lo), nm_hi = fmaxf(m_hi, bm_hi);
            if (__any_sync(0xffffffffu, nm_lo != m_lo || nm_hi != m_hi)) {
                const float corr_lo = ex2_approx(m_lo - nm_lo), corr_hi = ex2_approx(m_hi - nm_hi);
                m_lo = nm_lo; m_hi = nm_hi;
                l_lo *= corr_lo; l_hi *= corr_hi;
                acc[0] *= corr_lo; acc[1] *= corr_lo; acc[2] *= corr_hi; acc[3] *= corr_hi;
            }
            // P enters the P.V product as plain bf16: its rounding (2^-9 relative per weight, averaged over the keys) is far below
            // the bf16 rounding the attention OUTPUT receives anyway (att16 is the next GEMM's bf16 operand)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                uint32_t ph[4];
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) {
                    const float* c = sc[half * 2 + nt];
                    const float e0 = ex2_approx(c[0] - m_lo), e1 = ex2_approx(c[1] - m_lo);
                    const float e2 = ex2_approx(c[2] - m_hi), e3 = ex2_approx(c[3] - m_hi);
                    l_lo += e0 + e1; l_hi += e2 + e3;
                    const __nv_bfloat162 p01 = __floats2bfloat162_rn(e0, e1), p23 = __floats2bfloat162_rn(e2, e3);
                    ph[nt * 2] = *reinterpret_cast<const uint32_t*>(&p01);
                    ph[nt * 2 + 1] = *reinterpret_cast<const uint32_t*>(&p23);
                }
                const uint32_t* vr = reinterpret_cast<const uint32_t*>(Vt + (size_t)gq * vstride + kb + half * 16 + 2 * tq);
                mma_bf16_16816(acc, ph, vr[0], vr[4]);
            }
        }
        l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 1); l_lo += __shfl_xor_sync(0xffffffffu, l_lo, 2);
        l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 1); l_hi += __shfl_xor_sync(0xffffffffu, l_hi, 2);
        const int col = h * DH + 2 * tq;
        if (c_lo < nc) {
            const float o0 = acc[0] / l_lo, o1 = acc[1] / l_lo;
            if (out) *reinterpret_cast<float2*>(out + n_lo * D + col) = make_float2(o0, o1);
            if (out16) *reinterpret_cast<__nv_bfloat162*>(out16 + n_lo * D + col) = __floats2bfloat162_rn(o0, o1);
        }
        if (c_hi < nc) {
            const float o0 = acc[2] / l_hi, o1 = acc[3] / l_hi;
            if (out) *reinterpret_cast<float2*>(out + n_hi * D + col) = make_float2(o0, o1);
            if (out16) *reinterpret_cast<__nv_bfloat162*>(out16 + n_hi * D + col) = __floats2bfloat162_rn(o0, o1);
        }
    }
}

// ===========================================================================
// Fused vocab projection + softmax(logits / T) + greedy | multinomial pick
// (validate_generate_MMT_v15_4.py:753-759, 868-872).  One warp per sequence.
// ===========================================================================
struct SampleParams {
    const float* x;          // [N][D] decoder output of the newest position
    const float* W;          // fc_out.weight [V][D]
    const float* b;          // fc_out.bias [V]
    int V;
    int64_t N;               // sequences handled by this launch
    int64_t ldn;             // row length of tokens / probs / logits (sequences in the whole call)
    float temperature;
    int mode;                // 0 greedy, 1 multinomial, 2 forced (logits only)
    RngGeom rng;             // rng.offset is the offset of step 0; step t adds t*rng_inc
    uint64_t rng_inc;
    const uint64_t* rng_dev; // optional {seed, offset} in device memory (overrides rng.seed / rng.offset: keeps a captured
                             // decode graph reusable across calls with a different generator state)
    int64_t seq_index_base;
    int64_t rng_cand;        // 0: global mapping; > 0: per-memory streams of rng_cand rows, rng_col_steps calls per column
    int64_t rng_col_steps;   //   (torch_rng_row; rng.threads / rng_inc then describe one (rng_cand, V) call)
    int64_t* tokens;         // [max_len][N] or nullptr
    float* probs;            // [max_len][N] or nullptr
    float* logits;           // [T][N][V] (forced / unit test) or nullptr
    const int64_t* target;   // optional [max_len][N]: a token per sequence and position ...
    float* target_prob;      // ... whose softmax(logits / T) probability is written here (teacher-forced scorers)
    StepCtl ctl;             // ctl.step may be nullptr (stand-alone use, t = 0)
    int advance;             // 1: the last CTA increments *ctl.step
    // optional prologue (fused decoder path): x <- LN(x + pbias + sum_s part[s]) -- the last layer's FFN2 + norm3
    const float* part; int splits; int64_t part_stride;
    const float* pbias; const float* pgamma; const float* pbeta; float eps;
    int rows_per_warp;       // dense input: 1 or SAMPLE_NR rows per warp (0 = 1)
    // stop at <EOS> (mmt_decode_until_eos), all nullptr otherwise: row r is sequence orig[r] of the launch (compacted wave,
    // kernels_retire.cuh; nullptr = r), whose first-<EOS> step eos_len[] holds (max_len until it emits `eos`).  A
    // finished sequence writes <PAD> / 0 and counts as <PAD>; live[t] counts the sequences not finished after step t.
    const int* orig; int* eos_len; int* live; int64_t eos;
};

// CTA = 8 warps.  Rows are taken in groups of `rpc` per CTA, grid-stride: a CTA stages fc_out once and keeps sampling
// groups (large waves: 2048 CTAs each re-loading the 22 KB matrix cost more than the sampling itself).
// rpc = 32 (dense input): a warp owns FOUR rows and walks fc_out once for all of them -- with one row per warp the 43 x 128
// projection is 384 shared-memory loads per row (the kernel was bound by them: 173 us per position of 75,776 rows); four
// rows share every weight load and read x as broadcast float4 (96 per row).  Every accumulator still sums k = 0 .. 127 in
// order: the logits are bit-identical to the one-row form.
// rpc = 2 (fused decoder path, whose input is still spread over the FFN2 split partials): four warps per row in the input
// phase, each with a quarter of the partials in flight at once -- the reduction is an L2 round trip per pass, so its depth
// sets the kernel's latency on the 13-kernel chain of a small wave -- then one row per warp.
constexpr int SAMPLE_NR = 4;             // rows per warp (dense input)
constexpr int SAMPLE_ROWS = 8 * SAMPLE_NR;

template <int NR>
__device__ __forceinline__ void sample_rows(const SampleParams& p, const float* Ws, const float (*xs)[D], int r0, int64_t n0, int t, int lane, int& my_nonpad,
                                            int& my_live) {
    const int v0 = lane, v1 = lane + 32;
    float a0[NR], a1[NR];
#pragma unroll
    for (int r = 0; r < NR; ++r) { a0[r] = 0.f; a1[r] = 0.f; }
    const float* w0 = Ws + v0 * (D + 1);
    const float* w1 = Ws + (v1 < p.V ? v1 : 0) * (D + 1);
#pragma unroll 2
    for (int k = 0; k < D; k += 4) {
        const float w00 = w0[k], w01 = w0[k + 1], w02 = w0[k + 2], w03 = w0[k + 3];
        const float w10 = w1[k], w11 = w1[k + 1], w12 = w1[k + 2], w13 = w1[k + 3];
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const float4 xv = *reinterpret_cast<const float4*>(&xs[r0 + r][k]);
            a0[r] = fmaf(xv.x, w00, a0[r]); a1[r] = fmaf(xv.x, w10, a1[r]);
            a0[r] = fmaf(xv.y, w01, a0[r]); a1[r] = fmaf(xv.y, w11, a1[r]);
            a0[r] = fmaf(xv.z, w02, a0[r]); a1[r] = fmaf(xv.z, w12, a1[r]);
            a0[r] = fmaf(xv.w, w03, a0[r]); a1[r] = fmaf(xv.w, w13, a1[r]);
        }
    }
    const bool ok0 = v0 < p.V, ok1 = v1 < p.V;
    const float b0 = ok0 ? p.b[v0] : 0.f, b1 = ok1 ? p.b[v1] : 0.f;
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const int64_t n = n0 + r;
        if (n >= p.N) break;
        const int64_t no = p.orig ? p.orig[n] : n;        // the sequence's own column and Philox row
        float lg0 = ok0 ? a0[r] + b0 : MMT_NEG_INF;
        float lg1 = ok1 ? a1[r] + b1 : MMT_NEG_INF;
        if (p.logits) {
            float* out = p.logits + ((int64_t)t * p.ldn + n) * p.V;
            if (ok0) out[v0] = lg0;
            if (ok1) out[v1] = lg1;
        }
        if (p.mode == 2) continue;
        float z0 = ok0 ? lg0 / p.temperature : MMT_NEG_INF;
        float z1 = ok1 ? lg1 / p.temperature : MMT_NEG_INF;
        float mx = warp_max(fmaxf(z0, z1));
        float e0 = ok0 ? expf(z0 - mx) : 0.f;
        float e1 = ok1 ? expf(z1 - mx) : 0.f;
        float sum = warp_sum(e0 + e1);
        float p0 = e0 / sum, p1 = e1 / sum;
        if (p.target) {       // probability of the given token (validate_generate_MMT_v15_4.py:372-374)
            const int64_t tg = p.target[(int64_t)t * p.ldn + n];
            const float a = __shfl_sync(0xffffffffu, p0, (int)(tg & 31)), b = __shfl_sync(0xffffffffu, p1, (int)(tg & 31));
            if (lane == 0) p.target_prob[(int64_t)t * p.ldn + n] = (tg < 0 || tg >= p.V) ? 0.f : (tg < 32 ? a : b);
        }
        float r0v = p0, r1v = p1;
        if (p.mode == 1) {
            RngGeom g = p.rng;
            if (p.rng_dev) { g.seed = p.rng_dev[0]; g.offset = p.rng_dev[1]; }
            const int64_t li = torch_rng_row(g, p.rng_inc, p.rng_cand, p.rng_col_steps, p.seq_index_base + no, t, p.V);
            if (ok0) r0v = p0 / torch_exponential_at(g, li + v0);
            if (ok1) r1v = p1 / torch_exponential_at(g, li + v1);
        }
        // argmax with lowest-index ties (torch argmax / multinomial)
        float best = ok0 ? r0v : MMT_NEG_INF;
        int bi = ok0 ? v0 : 0x7fffffff;
        float bp = p0;
        if (ok1 && (r1v > best)) { best = r1v; bi = v1; bp = p1; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            float ob = __shfl_xor_sync(0xffffffffu, best, o);
            int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            float op = __shfl_xor_sync(0xffffffffu, bp, o);
            if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; bp = op; }
        }
        if (lane == 0) {
            bool fin = false;
            if (p.eos_len) {
                fin = t > p.eos_len[no];
                if (!fin && bi == p.eos) p.eos_len[no] = t;
                my_live += !fin && bi != p.eos;
            }
            if (p.tokens) p.tokens[(int64_t)t * p.ldn + no] = fin ? 0 : bi;
            if (p.probs) p.probs[(int64_t)t * p.ldn + no] = fin ? 0.f : bp;
            my_nonpad += !fin && bi != 0;
        }
    }
}

// dynamic shared memory: fc_out as V padded rows (sample_smem_bytes)
__host__ __device__ constexpr size_t sample_smem_bytes(int V) { return (size_t)V * (D + 1) * sizeof(float); }
__global__ void __launch_bounds__(256) sample_tokens(const __grid_constant__ SampleParams p) {
    extern __shared__ float Ws[];
    __shared__ __align__(16) float xs[SAMPLE_ROWS][D];
    __shared__ __align__(16) float psum[8][D];
    __shared__ int s_nonpad, s_live;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    pdl_launch_dependents();
    // fc_out weights -> padded smem rows (independent of the step: issued before anything else)
    for (int i = threadIdx.x; i < p.V * (D / 4); i += blockDim.x) {
        const float4 w = *reinterpret_cast<const float4*>(p.W + (int64_t)i * 4);
        float* dst = Ws + (i / (D / 4)) * (D + 1) + (i % (D / 4)) * 4;
        dst[0] = w.x; dst[1] = w.y; dst[2] = w.z; dst[3] = w.w;
    }
    if (threadIdx.x == 0) { s_nonpad = 0; s_live = 0; }
    pdl_wait();
    const int t = p.ctl.step ? *p.ctl.step : 0;
    const bool nr4 = p.rows_per_warp == SAMPLE_NR;
    const int rpc = p.part ? 2 : (nr4 ? SAMPLE_ROWS : 8);       // rows per CTA and pass
    int my_nonpad = 0, my_live = 0;
    for (int64_t base = (int64_t)blockIdx.x * rpc; base < p.N; base += (int64_t)gridDim.x * rpc) {
        if (p.part) {   // ---- input rows -> xs: four warps per row over the FFN2 partials
            const int wpr = 4;
            const int r = warp / wpr, sl = warp % wpr;
            const int64_t n = base + r;
            if (n < p.N) {
                // slice sl sums partials sl, sl + wpr, ... (all in flight together), fixed order
                float4 q[8];
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int k0 = sl; k0 < p.splits; k0 += 8 * wpr) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) {
                        const int k = k0 + u * wpr;
                        q[u] = (k < p.splits) ? *reinterpret_cast<const float4*>(p.part + (int64_t)k * p.part_stride + n * D + lane * 4)
                                              : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int u = 0; u < 8; ++u) { a.x += q[u].x; a.y += q[u].y; a.z += q[u].z; a.w += q[u].w; }
                }
                *reinterpret_cast<float4*>(&psum[warp][lane * 4]) = a;
            }
            __syncthreads();
            if (warp < rpc && base + warp < p.N) {   // x <- LN3(x + b2 + sum of the slices), slices in fixed order
                const int64_t n2 = base + warp;
                float4 v = *reinterpret_cast<const float4*>(p.x + n2 * D + lane * 4);
                float4 sum = *reinterpret_cast<const float4*>(p.pbias + lane * 4);
                for (int j = 0; j < wpr; ++j) {
                    const float4 q = *reinterpret_cast<const float4*>(&psum[warp * wpr + j][lane * 4]);
                    sum.x += q.x; sum.y += q.y; sum.z += q.z; sum.w += q.w;
                }
                v = ln_row(make_float4(v.x + sum.x, v.y + sum.y, v.z + sum.z, v.w + sum.w), p.pgamma, p.pbeta, p.eps, lane);
                *reinterpret_cast<float4*>(&xs[warp][lane * 4]) = v;
            }
            __syncthreads();
            if (warp < rpc && base + warp < p.N) sample_rows<1>(p, Ws, xs, warp, base + warp, t, lane, my_nonpad, my_live);
        } else if (nr4) {   // ---- dense input: each warp stages and samples its own four rows
#pragma unroll
            for (int r = 0; r < SAMPLE_NR; ++r) {
                const int64_t n = base + warp * SAMPLE_NR + r;
                if (n < p.N) *reinterpret_cast<float4*>(&xs[warp * SAMPLE_NR + r][lane * 4]) = *reinterpret_cast<const float4*>(p.x + n * D + lane * 4);
            }
            __syncthreads();      // (also orders the Ws staging of the first pass)
            if (base + warp * SAMPLE_NR < p.N) sample_rows<SAMPLE_NR>(p, Ws, xs, warp * SAMPLE_NR, base + warp * SAMPLE_NR, t, lane, my_nonpad, my_live);
        } else {            // ---- dense input, small waves: one row per warp (more CTAs, shorter chain)
            const int64_t n = base + warp;
            if (n < p.N) *reinterpret_cast<float4*>(&xs[warp][lane * 4]) = *reinterpret_cast<const float4*>(p.x + n * D + lane * 4);
            __syncthreads();
            if (n < p.N) sample_rows<1>(p, Ws, xs, warp, n, t, lane, my_nonpad, my_live);
        }
        __syncthreads();          // xs / psum are rewritten by the next group
    }
    if (p.advance || p.ctl.nonpad || p.live) {
        if (my_nonpad) atomicAdd(&s_nonpad, my_nonpad);
        if (my_live) atomicAdd(&s_live, my_live);
        __syncthreads();
        if (threadIdx.x == 0) {   // one global atomic per CTA, not per sequence
            if (p.ctl.nonpad && s_nonpad) atomicAdd(p.ctl.nonpad + t, s_nonpad);
            if (p.live && s_live) atomicAdd(p.live + t, s_live);
            if (p.advance) {
                __threadfence();
                int done = atomicAdd(p.ctl.done_ctas, 1);
                if (done == (int)gridDim.x - 1) {
                    *p.ctl.done_ctas = 0;
                    *p.ctl.step = t + 1;
                }
            }
        }
    }
}

// q[i] = the Exp(1) variate torch's exponential_ writes at linear element base + i (unit-test hook, mmt_exponential)
__global__ void __launch_bounds__(256) exponential_fill(RngGeom g, int64_t base, int64_t n, float* q) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) q[i] = torch_exponential_at(g, base + i);
}

// token[n] = first arg-max over v of p[n][v] / q[li + v]   (torch.multinomial(p, 1) on given probabilities), li and the
// offset of row seq_base + n at step t from torch_rng_row (n_cand == 0, t == 0: element (seq_base + n) * V, offset g.offset)
__global__ void __launch_bounds__(256) sample_from_probs(const float* p, int64_t N, int V, RngGeom g, int64_t seq_base, uint64_t inc,
                                                         int64_t n_cand, int64_t col_steps, int t, int64_t* token) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t n = (int64_t)blockIdx.x * 8 + warp;
    if (n >= N) return;
    const int64_t li = torch_rng_row(g, inc, n_cand, col_steps, seq_base + n, t, V);
    float best = MMT_NEG_INF;
    int bi = 0x7fffffff;
    for (int v = lane; v < V; v += 32) {
        const float r = p[n * V + v] / torch_exponential_at(g, li + v);
        if (r > best) { best = r; bi = v; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
    }
    if (lane == 0) token[n] = bi;
}

// len[n] = index of the first `eos` in column n of tokens (T, N), or T when there is none
// (the truncation rule of helper_functions_pl_v15_4.py:272-301, 390-419).  One thread per sequence; rows are
// contiguous over n, so every step of the scan is a coalesced read.
__global__ void first_eos_scan(const int64_t* tokens, int T, int64_t N, int eos, int32_t* len) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    int L = T;
    for (int t = 0; t < T; ++t)
        if (tokens[(int64_t)t * N + n] == eos) { L = t; break; }
    len[n] = L;
}

// Ragged ingest (reference dataloaders_pl_v15_4.py:267-299 _zero_pad, :352-365 / :456-460 / :481-485 normalisation):
// CSR peak lists -> the padded (B,P[,cols]) fp32 tensor + (B,P) mask of the collate contract.  Values are divided in
// double like the reference's Python floats, then rounded to fp32 (torch.tensor of Python floats).  Peaks beyond P are
// dropped.  `quirk_1d`: the reference's 1-D branch leaves the mask all-ones when a list has >= P entries (SURVEY A.1).
__global__ void __launch_bounds__(64) ingest_peaks(const double* vals, const int64_t* off, int cols, double div0, double div1,
                                                   int P, int quirk_1d, float* src, float* mask) {
    const int b = blockIdx.x;
    const int64_t o = off[b];
    const int64_t n = off[b + 1] - o;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const bool have = i < n;
        for (int c = 0; c < cols; ++c)
            src[((int64_t)b * P + i) * cols + c] = have ? (float)(vals[(o + i) * cols + c] / (c == 0 ? div0 : div1)) : 0.f;
        mask[(int64_t)b * P + i] = (quirk_1d && n >= P) ? 1.f : (have ? 0.f : 1.f);
    }
}

// IR spectrum -> `bins` mean-binned, max-normalised values (dataloaders_pl_v15_4.py:324-346): bin i averages
// spectra[round(start_i) : round(start_i + span)] with span = len / bins, start accumulated in double exactly like the
// reference's loop (Python round = round-half-even = rint), divided by the spectrum's maximum.
__global__ void __launch_bounds__(256) ingest_ir(const double* vals, const int64_t* off, int bins, float* out) {
    extern __shared__ int ir_edges[];          // [bins + 1]
    __shared__ double red[256];
    const int b = blockIdx.x;
    const double* x = vals + off[b];
    const int64_t len = off[b + 1] - off[b];
    double mx = -INFINITY;
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) mx = fmax(mx, x[i]);
    red[threadIdx.x] = mx;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) { if (threadIdx.x < s) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + s]); __syncthreads(); }
    mx = red[0];
    if (threadIdx.x == 0) {
        const double span = (double)len / (double)bins;
        double start = 0.0;
        for (int i = 0; i < bins; ++i) { ir_edges[i] = (int)rint(start); start = start + span; }
        ir_edges[bins] = (int)rint(start);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < bins; i += blockDim.x) {
        // slice [round(start_i), round(end_i)) with end_i = start_i + span = start_{i+1} (same double)
        const int64_t lo = min((int64_t)ir_edges[i], len), hi = min((int64_t)ir_edges[i + 1], len);
        double sum = 0.0;
        for (int64_t k = lo; k < hi; ++k) sum += x[k];
        out[(int64_t)b * bins + i] = (float)((sum / (double)(hi - lo)) / mx);      // empty slice -> NaN like np.mean([])
    }
}

// Bitwise comparison of up to 16 pairs of arrays (the collated inputs of two encode calls): *differ |= 1 on any mismatch.
struct CompareParams { const unsigned char* a[16]; const unsigned char* b[16]; int64_t bytes[16]; int n; int* differ; };
__global__ void __launch_bounds__(256) compare_segments(const __grid_constant__ CompareParams p) {
    const int sgm = blockIdx.y;
    const unsigned char *x = p.a[sgm], *y = p.b[sgm];
    const int64_t nb = p.bytes[sgm];
    bool diff = false;
    if ((((uintptr_t)x | (uintptr_t)y | (uintptr_t)nb) & 15) == 0) {
        const uint4 *x4 = reinterpret_cast<const uint4*>(x), *y4 = reinterpret_cast<const uint4*>(y);
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb / 16; i += (int64_t)gridDim.x * blockDim.x) {
            const uint4 u = x4[i], v = y4[i];
            diff |= (u.x != v.x) | (u.y != v.y) | (u.z != v.z) | (u.w != v.w);
        }
    } else {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += (int64_t)gridDim.x * blockDim.x) diff |= x[i] != y[i];
    }
    if (__syncthreads_or(diff) && threadIdx.x == 0) atomicOr(p.differ, 1);
}

__global__ void set_u64x2(uint64_t* dst, uint64_t a, uint64_t b) { dst[0] = a; dst[1] = b; }

__global__ void pack_tokens_u8(const int64_t* in, int64_t n, uint8_t* out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (uint8_t)in[i];
}
__global__ void unpack_tokens_u8(const uint8_t* in, int64_t n, int64_t* out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int64_t)in[i];
}
// (T,N) i64 -> (N,T) u8 and (N,T) u8 -> (T,N) i64: 32 x 32 tiles through shared memory, both sides coalesced
__global__ void __launch_bounds__(256) pack_tokens_u8_seqmajor(const int64_t* in, int T, int64_t N, uint8_t* out) {
    __shared__ uint8_t tile[32][33];
    const int64_t n0 = (int64_t)blockIdx.x * 32;
    const int t0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8)
        if (t0 + r < T && n0 + tx < N) tile[r][tx] = (uint8_t)in[(int64_t)(t0 + r) * N + n0 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8)
        if (n0 + r < N && t0 + tx < T) out[(n0 + r) * T + t0 + tx] = tile[tx][r];
}
__global__ void __launch_bounds__(256) unpack_tokens_u8_seqmajor(const uint8_t* in, int T, int64_t N, int64_t* out) {
    __shared__ uint8_t tile[32][33];
    const int64_t n0 = (int64_t)blockIdx.x * 32;
    const int t0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int r = ty; r < 32; r += 8)
        if (n0 + r < N && t0 + tx < T) tile[r][tx] = in[(n0 + r) * T + t0 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8)
        if (t0 + r < T && n0 + tx < N) out[(int64_t)(t0 + r) * N + n0 + tx] = (int64_t)tile[tx][r];
}
__global__ void f32_to_bf16(const float* in, int64_t n, __nv_bfloat16* out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __float2bfloat16_rn(in[i]);
}

__global__ void bf16_to_f32(const __nv_bfloat16* in, int64_t n, float* out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __bfloat162float(in[i]);
}

__global__ void set_i32(int* dst, int v) { *dst = v; }

}  // namespace mmt
