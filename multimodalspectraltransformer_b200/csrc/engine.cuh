// Host-side engine state: weight registry, workspace arena, launch helpers.
#pragma once
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/mmt_b200.h"
#include "common.cuh"

namespace mmt {

extern thread_local std::string g_last_error;

#define MMT_FAIL(msg)                                                                   \
    do {                                                                                \
        ::mmt::g_last_error = std::string(__FILE__) + ":" + std::to_string(__LINE__) + ": " + (msg); \
        return 1;                                                                       \
    } while (0)
#define MMT_CUDA(call)                                                                  \
    do {                                                                                \
        cudaError_t err__ = (call);                                                     \
        if (err__ != cudaSuccess) MMT_FAIL(std::string(#call) + " -> " + cudaGetErrorString(err__)); \
    } while (0)
#define MMT_TRY(call)                                                                   \
    do {                                                                                \
        if ((call) != 0) return 1;                                                      \
    } while (0)

struct Slot { std::string name; int64_t numel; int64_t off; };

struct Registry {
    std::vector<Slot> slots;
    std::unordered_map<std::string, int> index;
    int64_t total = 0;
    void add(const std::string& name, int64_t numel) {
        // every tensor starts on a 64-element boundary (256 B in the fp32 blob, 128 B in the
        // bf16 copy: vector loads and TMA descriptors need 16-byte aligned bases)
        index[name] = (int)slots.size();
        slots.push_back({name, numel, total});
        total += (numel + 63) / 64 * 64;
    }
};

inline Registry build_registry(const mmt_model_desc& d) {
    Registry r;
    const int64_t h = d.d_model, F = d.d_ff;
    auto lin = [&](const std::string& p, int64_t out, int64_t in) { r.add(p + ".weight", out * in); r.add(p + ".bias", out); };
    lin("linear_spec_embedding_1H.point_embedding_layer_1H.fc_H", h, 2);
    lin("linear_spec_embedding_13C.point_embedding_layer_13C.fc_C", h, 1);
    lin("linear_spec_embedding_HSQC.point_embedding_layer_HSQC.fc_HSQC", h, 2);
    lin("linear_spec_embedding_COSY.point_embedding_layer_COSY.fc_COSY", h, 2);
    lin("linear_spec_embedding_IR.linear_spec_embedding_IR", h, d.ir_bins);
    r.add("linear_embedding_MF.embedding.weight", (int64_t)d.mf_vocab * h);
    r.add("linear_embedding_MS.embedding.weight", (int64_t)d.ms_vocab * h);
    lin("linear_embedding_MW.linear_spec_embedding_MW", h, 1);
    r.add("embed_trg.weight", (int64_t)d.vocab * h);
    r.add("pe_trg.weight", (int64_t)d.max_len * h);
    auto attn = [&](const std::string& p) {
        r.add(p + ".in_proj_weight", 3 * h * h); r.add(p + ".in_proj_bias", 3 * h);
        lin(p + ".out_proj", h, h);
    };
    auto norm = [&](const std::string& p) { r.add(p + ".weight", h); r.add(p + ".bias", h); };
    const char* encs[6] = {"encoder_1H", "encoder_13C", "encoder_HSQC", "encoder_COSY", "encoder_IR", "encoder_cross"};
    for (const char* e : encs)
        for (int l = 0; l < d.n_enc_layers; ++l) {
            std::string p = std::string(e) + ".layers." + std::to_string(l);
            attn(p + ".self_attn");
            lin(p + ".linear1", F, h); lin(p + ".linear2", h, F);
            norm(p + ".norm1"); norm(p + ".norm2");
        }
    for (int l = 0; l < d.n_dec_layers; ++l) {
        std::string p = "decoder.layers." + std::to_string(l);
        attn(p + ".self_attn"); attn(p + ".multihead_attn");
        lin(p + ".linear1", F, h); lin(p + ".linear2", h, F);
        norm(p + ".norm1"); norm(p + ".norm2"); norm(p + ".norm3");
    }
    lin("fp1", d.fp_size, h);
    lin("fc_out", d.vocab, h);
    lin("real_data_linear", d.vocab, h);
    return r;
}

struct LayerW {   // fp32 pointers into the device blob
    const float *in_w, *in_b, *out_w, *out_b;        // self attention
    const float *ca_in_w, *ca_in_b, *ca_out_w, *ca_out_b;   // decoder cross attention
    const float *l1_w, *l1_b, *l2_w, *l2_b;
    const float *n1_w, *n1_b, *n2_w, *n2_b, *n3_w, *n3_b;
};

// Bump allocator over one grow-only device arena; `plan` mode only measures.
struct Arena {
    char* base = nullptr;
    size_t cap = 0, off = 0;
    bool plan = true;
    template <typename T>
    T* get(size_t n) {
        size_t bytes = (n * sizeof(T) + 255) & ~size_t(255);
        T* p = plan ? nullptr : reinterpret_cast<T*>(base + off);
        off += bytes;
        return p;
    }
};

}  // namespace mmt

struct mmt_engine {
    mmt_model_desc desc;
    int device = 0, sm_count = 0, max_threads_per_sm = 0;
    size_t total_mem = 0;              // device memory (default decode wave size)
    mmt::Registry reg;
    float* w32 = nullptr;
    __nv_bfloat16* w16 = nullptr;      // bf16(w32)
    __nv_bfloat16* w16lo = nullptr;    // bf16(w32 - w16): low-order term of the two-term weight split
    std::vector<mmt::LayerW> enc[6];   // 5 modality stacks + cross
    std::vector<mmt::LayerW> dec;
    char* arena = nullptr;
    size_t arena_bytes = 0;
    int64_t launches = 0;
    bool use_graph = true;             // replay the decode step as a CUDA graph (MMT_NO_GRAPH=1 disables)
    int fused_decode_rows = 2048;      // waves of at most this many sequences take the fused row-local decoder kernels (MMT_FUSED_DECODE_ROWS overrides; 0 disables)
    int max_wave_seqs = 0;             // sequences decoded together; larger runs go wave by wave (bounds the self-attention KV pool); 0 = default by precision (MMT_MAX_WAVE_SEQS overrides)
    bool enc_ffn_single = false;       // experiment (MMT_ENC_FFN_SINGLE=1): encoder FFN with the hi weight term only
    bool use_ffn_prologue = true;      // un-fused decode step, >= 2048 rows: cross-attention out-projection + norm2 inside the FFN kernel (MMT_NO_FFN_PROLOGUE=1 disables)
    bool use_cluster_ffn = false;      // MMT_CLUSTER_FFN=1: small bf16 waves run the FFN inside decode_attn, launched as clusters of 4 CTAs (parity-tested; measured equal to the separate fused-FFN kernel in the bench, profiles/r02_cluster_probe.md)
    bool kv_tok_major = true;          // un-fused bf16 step with the KV epilogue: token-major cache pages + decode_self_attention_tm (MMT_KV_HEAD_MAJOR=1: head-major pages + decode_self_attention_g8)
    bool use_l0_table = true;          // un-fused bf16 token-major step: decoder layer 0's Q / K | V from the position x token table (MMT_NO_L0_TABLE=1: the paged cache like layers 1-5)
    float* l0_qtab = nullptr;          // that table (built at the first decode that uses it): Q [pos][tok][D] fp32
    __nv_bfloat16* l0_kvtab = nullptr; //   and K | V [pos][tok][2 D] bf16
    bool use_kv_epilogue = true;       // un-fused bf16 step: the QKV projection's epilogue writes K | V of the new position into the cache pages (MMT_NO_KV_EPILOGUE=1: the attention kernel appends)
    bool use_ffn_wide = true;          // hi-term FFN with the LayerNorm epilogue: 128-column chunks (MMT_NO_FFN_WIDE=1: 64)
    bool use_gemm_chain = true;        // un-fused decode step: out-proj + LN1 + cross-attention query projection as one launch (MMT_NO_GEMM_CHAIN=1 disables)
    bool dec_proj_single = true;       // un-fused bf16 step: attention projections on the hi weight term only (MMT_DEC_PROJ_TWO_TERM=1: both terms)
    bool sample_ready = false;         // sample_tokens' dynamic shared memory attribute set
    bool dec_ffn_single = true;        // decoder FFN on the hi weight term only (MMT_DEC_FFN_TWO_TERM=1: both terms)
    bool use_compact = true;           // ragged encoder: compute distinct token rows only (MMT_DENSE_ENCODER=1 disables)
    struct GraphEntry { std::vector<uint64_t> key; cudaGraphExec_t exec; int64_t launches_per_group; uint64_t stamp; };
    std::vector<GraphEntry> graph_cache;   // instantiated decode-step graphs of single-wave runs (staged outputs), keyed by what their nodes bake in
    uint64_t graph_cache_clock = 0;
    bool use_graph_cache = true;           // MMT_NO_GRAPH_CACHE=1: capture + instantiate on every call, write the caller's tensors directly
    bool use_tc_attention = true;      // encoder_cross attention on mma.sync in the bf16 mode (MMT_NO_TC_ATTENTION=1: fp32 SIMT kernel)
    bool use_tc5_attention = false;    // encoder_cross attention on tcgen05 / TMEM instead of mma.sync (opt-in: MMT_TC5_ATTENTION=1; correct but slower at these shapes)
    bool tc_attention_fp32 = false;    // test hook (MMT_TC_ATTENTION_FP32=1): the same kernel in the fp32 check mode, where nothing downstream amplifies its round-off
    int ffn_splits_override = 0;       // experiment knob (MMT_FFN_SPLITS): F-splits of the fused decode step's FFN
    bool use_enc_streams = true;       // ragged encoder: the five modality stacks as concurrent chains (MMT_NO_ENC_STREAMS=1 disables)
    cudaStream_t enc_stream[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t enc_ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int graph_steps = 16;              // decode positions captured per CUDA graph (MMT_GRAPH_STEPS overrides)
    int pdl_rows = 4096;               // un-fused bf16 step: programmatic dependent launch through the kernel chain for waves up to this many rows (MMT_PDL_ROWS overrides)
    bool use_pdl = true;               // programmatic dependent launch between the kernels of a fused decode step (MMT_NO_PDL=1 disables)
    cudaStream_t cap_stream[4] = {nullptr, nullptr, nullptr, nullptr};   // capture-only streams, one per decode lane (the caller's stream may be the legacy default stream)
    cudaEvent_t lane_ev[4] = {nullptr, nullptr, nullptr, nullptr};       // fork / join events of the lane branches
    int decode_lanes = 2;              // concurrent lanes of a small decode wave (MMT_DECODE_LANES overrides)
    int decode_lanes_large = 1;        // concurrent lanes of a large (un-fused) bf16 wave (MMT_DECODE_LANES_LARGE overrides)
    long long* ffn_dbg = nullptr;      // MMT_FFN_DEBUG phase timestamps of the un-fused FFN (managed memory)
    long long* da_dbg = nullptr;       // MMT_DA_DEBUG phase timestamps (managed memory)
    bool da_ready = false;             // decode_attn shared-memory attribute set
    bool tc_ready = false;             // tcgen05 path initialised (driver entry point + smem attributes)
    cudaEvent_t poll_ev[2] = {nullptr, nullptr};   // early-exit polls, one group behind the launches
    int32_t* h_pinned = nullptr;       // small pinned staging buffer (early-exit poll)
    // per-kernel-class device timing (mmt_profile_enable / mmt_profile_report)
    struct ProfRecord { const char* name; cudaEvent_t a, b; double work; };
    bool profiling = false;
    std::pair<cudaEvent_t, cudaEvent_t> prof_open{nullptr, nullptr};
    std::vector<ProfRecord> prof_records;

    // Calls on one engine are serialised (one workspace arena, one pinned staging buffer, one graph cache): every C-ABI
    // entry that touches the engine holds `mu` for its duration, and a call issued on a different stream than the previous
    // one first waits (device side) for the event the previous call recorded at its end -- mmt::EngineCall in engine.cu.
    std::mutex mu;
    cudaEvent_t last_use = nullptr;
    cudaStream_t last_stream = nullptr;
    bool last_use_valid = false;

    const float* W(const std::string& name) const { return w32 + reg.slots.at(reg.index.at(name)).off; }
    const __nv_bfloat16* Wb(const float* p) const { return w16 + (p - w32); }
    const __nv_bfloat16* Wlo(const float* p) const { return w16lo + (p - w32); }
};
