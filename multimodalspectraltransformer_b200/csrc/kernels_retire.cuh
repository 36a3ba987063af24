// Retirement of finished sequences from a large decode wave (mmt_decode_until_eos).
//
// A wave's rows are compacted at group boundaries: the rows still live at the poll step t_poll (first <EOS> after
// t_poll, or none) are kept in their original order.  Row r of the compacted wave is sequence orig[r] of the lane; its
// KV pages are reached through the gathered block-table row, so no page moves.  Kept rows of one memory column stay
// contiguous: col_start / col_count give the candidate cross attention its rows per column.
#pragma once
#include "common.cuh"

// One CTA: stable scan of the keep flags eos_len[orig[r]] > t_poll over the M rows -> src[r'] = r (old row of new row r').
__global__ void __launch_bounds__(1024) retire_scan(const int* orig, const int* eos_len, int64_t M, int t_poll, int* src) {
    __shared__ int warp_tot[32];
    __shared__ int s_base;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int64_t r0 = 0; r0 < M; r0 += blockDim.x) {
        const int64_t r = r0 + threadIdx.x;
        const bool keep = r < M && eos_len[orig ? orig[r] : r] > t_poll;
        const unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) warp_tot[warp] = __popc(bal);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < warp; ++w) before += warp_tot[w];
        if (keep) src[before + __popc(bal & ((1u << lane) - 1u))] = (int)r;
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += warp_tot[w];
            s_base += tot;
        }
        __syncthreads();
    }
}

// New row r' < M_new: orig_new[r'] = orig[src[r']], block-table row gathered; per memory column (n_cand rows of the lane
// each) the first new row and the row count (col_count zeroed by the caller).
__global__ void __launch_bounds__(256) retire_gather(const int* src, const int* orig, const int* bt, int pps, int64_t M_new, int n_cand,
                                                     int* orig_new, int* bt_new, int* col_start, int* col_count) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= M_new) return;
    const int s = src[r];
    const int o = orig ? orig[s] : s;
    orig_new[r] = o;
    for (int j = 0; j < pps; ++j) bt_new[r * pps + j] = bt[(int64_t)s * pps + j];
    const int col = o / n_cand;
    const int prev = r > 0 ? (orig ? orig[src[r - 1]] : src[r - 1]) / n_cand : -1;
    if (prev != col) col_start[col] = (int)r;
    atomicAdd(col_count + col, 1);
}

// Caller-facing outputs of a retiring call: len[n] = first <EOS> position (max_len if none); ids / probabilities after it,
// and at positions from `steps` on, become <PAD> / 0.
__global__ void __launch_bounds__(256) retire_fill(int64_t* tokens, float* probs, int T, int64_t N, const int* eos_len, int steps,
                                                   int32_t* len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)T * N) return;
    const int t = (int)(i / N);
    const int64_t n = i % N;
    const int L = eos_len[n];
    if (t == 0 && len) len[n] = L;
    if (t > L || t >= steps) {
        tokens[i] = 0;
        if (probs) probs[i] = 0.f;
    }
}

__global__ void fill_i32(int* p, int64_t n, int v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
