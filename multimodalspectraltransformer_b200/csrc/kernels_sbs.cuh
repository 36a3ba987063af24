// Stochastic beam search (Kool, van Hoof & Welling, ICML 2019): k distinct sequences per memory column that are an exact
// sample without replacement from the decoder's ancestral-sampling distribution at the column's temperature.
//
// Same wave layout as the deterministic search (kernels_beam.cuh): the k slots of a column are k rows of one KV-cached
// decode wave, children inherit closed pages by block-table entry and copy the open page (beam_copy_pages).  Per step:
//   sbs_select  one CTA per column: softmax(logits / tau_b) exactly as sample_tokens computes it, Gumbel-perturbed
//               log-probabilities with torch's Exp(1) variates (per-memory streams), the children's keys conditioned
//               on their parent's key (double), a block-wide radix select of the k largest of up to k*V candidates,
//               then the new slots' phi, key, length, token history, probabilities, block table and copy plan.
// Slot state lives in the arena in two parities (read t & 1, write (t + 1) & 1): a slot copies its parent's history
// row from the other parity, so no CTA stages k x 128 histories in shared memory.  Past a slot's length, and past the
// step that last wrote the row, history and probabilities are 0 (<PAD> / 0.f): rows are zeroed once by sbs_init and
// every write covers positions 0..t.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace mmt {

constexpr int SBS_MAX = 128;        // slots per column
constexpr int SBS_THREADS = 256;

struct SbsParams {
    const float* logits;     // [Nw][V] logits of the newest position
    int V, K, T, eos, pps;
    int64_t Nw;              // slots of this wave (columns * K)
    const int* step;         // device step counter, already advanced by the sampler: t = *step - 1
    const float* temp;       // [columns of the wave] temperature of each column
    RngGeom rng;             // threads / numel of one (K, V) exponential_ call; seed / offset of step 0 from rng_dev
    uint64_t rng_inc;
    const uint64_t* rng_dev; // {seed, offset} (nullptr: rng.seed / rng.offset)
    int64_t col_base;        // global column index of CTA 0 (seq_index_base / K + first column of the wave)
    // slot state, [parity]: phi / key (log-probability, Gumbel key; -inf: empty slot), len (generated tokens, <EOS>
    // included), hist [Nw][T] token ids, probs [Nw][T] p of each token
    double* phi[2]; double* key[2]; int* len[2]; uint8_t* hist[2]; float* probs[2];
    int64_t* cur_tok;        // [Nw] input token of the next step
    int* block_table;        // [Nw][pps]
    int* copy_src; int* copy_dst;   // [Nw] page to copy for the next step (-1: none)
    int* unfinished;         // [T] selected slots still open after step t (early exit); may be nullptr
    float* p_out;            // optional [Nw][V]: softmax of the live slots' logits (unit test)
};

// root state in parity 0 (slot 0 of every column: [<SOS>], phi = key = 0; the others empty), parity 1 zeroed
__global__ void sbs_init(const SbsParams p, int sos) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= p.Nw) return;
    const bool root = n % p.K == 0;
    for (int a = 0; a < 2; ++a) {
        p.phi[a][n] = root && a == 0 ? 0.0 : -INFINITY;
        p.key[a][n] = root && a == 0 ? 0.0 : -INFINITY;
        p.len[a][n] = 0;
        for (int i = 0; i < p.T; ++i) { p.hist[a][n * p.T + i] = 0; p.probs[a][n * p.T + i] = 0.f; }
    }
    p.cur_tok[n] = sos;
    p.copy_src[n] = -1; p.copy_dst[n] = -1;
    for (int q = 0; q < p.pps; ++q) p.block_table[n * p.pps + q] = (int)(n * p.pps + q);
}

// order-preserving map of a double onto uint64 (larger key -> larger code; -inf lowest)
__device__ __forceinline__ unsigned long long sbs_code(double x) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__device__ __forceinline__ double warp_max_f64(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// log(1 - exp(x)), x <= 0 (Maechler's split; -inf at x = 0)
__device__ __forceinline__ double sbs_log1mexp(double x) {
    return x > -0.6931471805599453 ? log(-expm1(x)) : log1p(-exp(x));
}

// key of a child: G - max(0, v) - log1p(exp(-|v|)), v = G - Gh + log1mexp(Gh - Z) (the paper's appendix, stable form)
__device__ __forceinline__ double sbs_child_key(double G, double Gh, double Z) {
    const double v = G - Gh + sbs_log1mexp(Gh - Z);
    return G - fmax(0.0, v) - log1p(exp(-fabs(v)));
}

// dynamic shared memory: candidate keys (double) and probabilities (float), K * V each
__host__ __device__ constexpr size_t sbs_smem_bytes(int K, int V) { return (size_t)K * V * (sizeof(double) + sizeof(float)); }

__global__ void __launch_bounds__(SBS_THREADS) sbs_select(const __grid_constant__ SbsParams p) {
    extern __shared__ __align__(16) unsigned char sbs_smem[];
    const int K = p.K, V = p.V, T = p.T;
    const int nc = K * V;                                  // candidate c = parent rank * V + token (carried leaf: + 0)
    double* c_key = reinterpret_cast<double*>(sbs_smem);
    float* c_prob = reinterpret_cast<float*>(c_key + nc);
    __shared__ double s_phi[SBS_MAX];
    __shared__ int s_len[SBS_MAX], bt_old[SBS_MAX][8];
    __shared__ uint8_t s_leaf[SBS_MAX];
    __shared__ unsigned s_hist[256];
    __shared__ int s_scan[2][SBS_THREADS];
    __shared__ int s_sel[SBS_MAX], s_order[SBS_MAX];
    __shared__ double s_selkey[SBS_MAX];
    __shared__ int s_digit, s_rem, s_valid;

    const int t = *p.step - 1, rd = t & 1, wr = rd ^ 1;
    const int64_t n0 = (int64_t)blockIdx.x * K;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float tau = p.temp[blockIdx.x];

    // ---- parents
    if (threadIdx.x == 0) s_valid = 0;
    if (threadIdx.x < K) {
        const int r = threadIdx.x;
        const int L = p.len[rd][n0 + r];
        s_len[r] = L;
        s_phi[r] = p.phi[rd][n0 + r];
        s_leaf[r] = L >= T || (L > 0 && p.hist[rd][(n0 + r) * T + L - 1] == p.eos);
    }
    for (int i = threadIdx.x; i < K * p.pps; i += blockDim.x) bt_old[i / p.pps][i % p.pps] = p.block_table[n0 * p.pps + i];
    __syncthreads();

    // ---- candidates: a warp per parent
    RngGeom g = p.rng;
    if (p.rng_dev) { g.seed = p.rng_dev[0]; g.offset = p.rng_dev[1]; }
    int my_valid = 0;
    for (int r = warp; r < K; r += SBS_THREADS / 32) {
        const double G = p.key[rd][n0 + r];
        double* ck = c_key + r * V;
        if (G == -INFINITY || s_leaf[r]) {                 // empty: no candidate; leaf: itself, unchanged, at its position
            for (int i = lane; i < V; i += 32) ck[i] = (i == 0 && G != -INFINITY) ? G : -INFINITY;
            my_valid += lane == 0 && G != -INFINITY;
            continue;
        }
        // softmax(logits / tau) exactly as sample_rows computes it
        const float* lg = p.logits + (n0 + r) * V;
        const int v0 = lane, v1 = lane + 32;
        const bool ok0 = v0 < V, ok1 = v1 < V;
        const float z0 = ok0 ? lg[v0] / tau : MMT_NEG_INF, z1 = ok1 ? lg[v1] / tau : MMT_NEG_INF;
        const float mx = warp_max(fmaxf(z0, z1));
        const float e0 = ok0 ? expf(z0 - mx) : 0.f, e1 = ok1 ? expf(z1 - mx) : 0.f;
        const float sum = warp_sum(e0 + e1);
        const float p0 = e0 / sum, p1 = e1 / sum;
        // perturbed log-probabilities: element r * V + i of the column's (K, V) exponential_ call of step t
        RngGeom gr = g;
        const int64_t li = torch_rng_row(gr, p.rng_inc, K, T, (p.col_base + blockIdx.x) * K + r, t, V);
        const double phi = s_phi[r];
        const bool c0 = ok0 && p0 > 0.f, c1 = ok1 && p1 > 0.f;
        const double gh0 = c0 ? phi + log((double)p0) - log((double)torch_exponential_at(gr, li + v0)) : -INFINITY;
        const double gh1 = c1 ? phi + log((double)p1) - log((double)torch_exponential_at(gr, li + v1)) : -INFINITY;
        const double Z = warp_max_f64(fmax(gh0, gh1));
        if (ok0) { ck[v0] = c0 ? sbs_child_key(G, gh0, Z) : -INFINITY; c_prob[r * V + v0] = p0; }
        if (ok1) { ck[v1] = c1 ? sbs_child_key(G, gh1, Z) : -INFINITY; c_prob[r * V + v1] = p1; }
        if (p.p_out && ok0) p.p_out[(n0 + r) * V + v0] = p0;
        if (p.p_out && ok1) p.p_out[(n0 + r) * V + v1] = p1;
        my_valid += (int)c0 + (int)c1;
    }
    if (my_valid) atomicAdd(&s_valid, my_valid);
    __syncthreads();
    const int kk = min(K, s_valid);                        // slots that get a sequence

    // ---- radix select: code of the kk-th largest key, 8 bits per pass from the top
    unsigned long long prefix = 0, pmask = 0;
    if (threadIdx.x == 0) s_rem = kk;
    for (int shift = 56; shift >= 0 && kk > 0; shift -= 8) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s_hist[i] = 0;
        __syncthreads();
        for (int c = threadIdx.x; c < nc; c += blockDim.x) {
            const unsigned long long u = sbs_code(c_key[c]);
            if ((u & pmask) == prefix) atomicAdd(&s_hist[(u >> shift) & 255], 1u);
        }
        __syncthreads();
        if (warp == 0) {                                   // lane l holds digits 255 - 8l .. 248 - 8l
            unsigned h[8], tot = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) { h[j] = s_hist[255 - 8 * lane - j]; tot += h[j]; }
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned x = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += x;
            }
            const unsigned rem = (unsigned)s_rem, excl = incl - tot;
            if (excl < rem && rem <= incl) {
                unsigned acc = excl;
                for (int j = 0; j < 8; ++j) {
                    if (acc + h[j] >= rem) { s_digit = 255 - 8 * lane - j; s_rem = (int)(rem - acc); break; }
                    acc += h[j];
                }
            }
        }
        __syncthreads();
        prefix |= (unsigned long long)s_digit << shift;
        pmask |= 255ull << shift;
    }
    // keys above the threshold, then threshold ties in candidate order: kk selected
    const int need_eq = kk > 0 ? s_rem : 0, n_gt = kk - need_eq;
    const int chunk = (nc + SBS_THREADS - 1) / SBS_THREADS, c_lo = threadIdx.x * chunk, c_hi = min(nc, c_lo + chunk);
    int n_g = 0, n_e = 0;
    if (kk > 0)
        for (int c = c_lo; c < c_hi; ++c) { const unsigned long long u = sbs_code(c_key[c]); n_g += u > prefix; n_e += u == prefix; }
    s_scan[0][threadIdx.x] = n_g; s_scan[1][threadIdx.x] = n_e;
    __syncthreads();
    if (warp < 2) {                                        // exclusive scans (warp 0: above, warp 1: ties), 8 per lane
        int* a = s_scan[warp];
        int v[SBS_THREADS / 32], tot = 0;
#pragma unroll
        for (int j = 0; j < SBS_THREADS / 32; ++j) { v[j] = a[lane * (SBS_THREADS / 32) + j]; tot += v[j]; }
        int incl = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int x = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += x;
        }
        int run = incl - tot;
#pragma unroll
        for (int j = 0; j < SBS_THREADS / 32; ++j) { a[lane * (SBS_THREADS / 32) + j] = run; run += v[j]; }
    }
    __syncthreads();
    if (kk > 0) {
        int pg_ = s_scan[0][threadIdx.x], pe = s_scan[1][threadIdx.x];
        for (int c = c_lo; c < c_hi; ++c) {
            const unsigned long long u = sbs_code(c_key[c]);
            if (u > prefix) s_sel[pg_++] = c;
            else if (u == prefix) { if (pe < need_eq) s_sel[n_gt + pe] = c; ++pe; }
        }
    }
    __syncthreads();
    // order of the kk selected: key descending, lower candidate first on equal keys
    if (threadIdx.x < kk) s_selkey[threadIdx.x] = c_key[s_sel[threadIdx.x]];
    __syncthreads();
    if (threadIdx.x < kk) {
        const int j = threadIdx.x, cj = s_sel[j];
        const double kj = s_selkey[j];
        int rank = 0;
        for (int i = 0; i < kk; ++i) rank += s_selkey[i] > kj || (s_selkey[i] == kj && s_sel[i] < cj);
        s_order[rank] = cj;
    }
    __syncthreads();

    // ---- new state of the K slots
    const int pg = t / PAGE_TOKENS, r16 = t % PAGE_TOKENS;
    int open = 0;
    if (threadIdx.x < K) {
        const int j = threadIdx.x;
        const int64_t n = n0 + j;
        if (j < kk) {
            const int c = s_order[j], q = c / V, tok = s_leaf[q] ? -1 : c % V;
            p.len[wr][n] = s_len[q] + (tok >= 0);
            p.phi[wr][n] = tok >= 0 ? s_phi[q] + log((double)c_prob[c]) : s_phi[q];
            p.key[wr][n] = c_key[c];
            p.cur_tok[n] = tok >= 0 ? tok : p.eos;
            open = tok >= 0 && tok != p.eos;
            for (int pp = 0; pp < pg; ++pp) p.block_table[n * p.pps + pp] = bt_old[q][pp];
            if (pg < p.pps) {
                if (r16 == PAGE_TOKENS - 1) {             // the page just closed: inherit it, the next page starts empty
                    p.block_table[n * p.pps + pg] = bt_old[q][pg];
                    p.copy_src[n] = -1; p.copy_dst[n] = -1;
                } else {
                    const int dst = (int)((((int64_t)wr) * p.Nw + n) * p.pps + pg);
                    p.block_table[n * p.pps + pg] = dst;
                    p.copy_src[n] = bt_old[q][pg]; p.copy_dst[n] = dst;
                }
            }
        } else {                                           // empty (it always was: its own pages are nobody else's)
            p.len[wr][n] = 0;
            p.phi[wr][n] = -INFINITY;
            p.key[wr][n] = -INFINITY;
            p.cur_tok[n] = 0;
            for (int pp = 0; pp < p.pps; ++pp) p.block_table[n * p.pps + pp] = (int)(n * p.pps + pp);
            p.copy_src[n] = -1; p.copy_dst[n] = -1;
        }
    }
    // histories and probabilities, positions 0..t (later ones are 0 in both parities)
    const int W = min(t + 1, T);
    for (int i = threadIdx.x; i < K * W; i += blockDim.x) {
        const int j = i / W, pos = i % W;
        uint8_t h = 0;
        float pr = 0.f;
        if (j < kk) {
            const int c = s_order[j], q = c / V, L = s_len[q];
            const int64_t src = (n0 + q) * T + pos;
            if (pos < L) { h = p.hist[rd][src]; pr = p.probs[rd][src]; }
            else if (pos == L && !s_leaf[q]) { h = (uint8_t)(c % V); pr = c_prob[c]; }
        }
        p.hist[wr][(n0 + j) * T + pos] = h;
        p.probs[wr][(n0 + j) * T + pos] = pr;
    }
    const int n_open = __syncthreads_count(open);
    if (threadIdx.x == 0 && n_open && p.unfinished) atomicAdd(p.unfinished + t, n_open);
}

// the call's outputs from the final state (parity = steps run): tokens / probs (T, ldn) at column n_base + n, length,
// log-probability, key
__global__ void sbs_finish(const SbsParams p, int64_t n_base, int64_t ldn, int64_t* tokens, float* probs, int32_t* len,
                           double* log_prob, double* key) {
    const int a = *p.step & 1;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.Nw * p.T) return;
    const int64_t pos = i / p.Nw, n = i % p.Nw;          // (position, slot): coalesced output rows
    tokens[pos * ldn + n_base + n] = p.hist[a][n * p.T + pos];
    probs[pos * ldn + n_base + n] = p.probs[a][n * p.T + pos];
    if (pos == 0) {
        len[n_base + n] = p.len[a][n];
        log_prob[n_base + n] = p.phi[a][n];
        key[n_base + n] = p.key[a][n];
    }
}

}  // namespace mmt
