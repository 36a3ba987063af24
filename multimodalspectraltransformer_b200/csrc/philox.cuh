// Philox4x32-10 counter RNG, laid out so that the fused sampler draws exactly the
// numbers torch.multinomial(p, 1) draws on CUDA for the same generator state.
//
// torch.multinomial(p,1) == argmax(p / q), q = empty_like(p).exponential_(1)
// (ATen Distributions multinomial fast path).  exponential_ on CUDA is
// distribution_elementwise_grid_stride_kernel (ATen/native/cuda/DistributionTemplates.h):
//   block 256, grid = min(SMs * (maxThreadsPerSM/256), ceil(numel/256)), unroll 4;
//   thread idx: curand_init(seed, /*subsequence*/ idx, offset) (curandStatePhilox4_32_10);
//   loop iteration `it` draws curand_uniform4 and element
//   li = idx + threads*(4*it + c) takes component c, transformed by -log(u)
//   with the u ~ 1 guard of ATen/core/TransformationHelper.h.
// With offset a multiple of 4 (torch only ever advances by multiples of 4) the
// float4 of iteration `it` is Philox4x32-10(counter = {offset/4 + it, subsequence}, key = seed).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace mmt {

struct RngGeom {            // launch geometry of the torch kernel being reproduced
    uint64_t seed;
    uint64_t offset;        // generator offset of this call (multiple of 4)
    int64_t  threads;       // 256 * grid
    int64_t  numel;         // N_total * vocab
};

__host__ __device__ inline int64_t torch_rng_threads(int64_t numel, int sm_count, int max_threads_per_sm) {
    const int64_t block = 256;
    int64_t grid = (numel + block - 1) / block;
    int64_t cap = (int64_t)sm_count * (max_threads_per_sm / block);
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    return grid * block;
}

__host__ __device__ inline uint64_t torch_rng_increment(int64_t numel, int sm_count, int max_threads_per_sm) {
    int64_t threads = torch_rng_threads(numel, sm_count, max_threads_per_sm);
    return (uint64_t)(((numel - 1) / (threads * 4) + 1) * 4);
}

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0;
        k.y += W1;
    }
    return c;
}

// Exp(1) variate torch would have written at linear index `li` of the q tensor.
__device__ __forceinline__ float torch_exponential_at(const RngGeom& g, int64_t li) {
    int64_t per_iter = g.threads * 4;
    int64_t it = li / per_iter;
    int64_t rem = li - it * per_iter;
    int comp = (int)(rem / g.threads);
    uint64_t idx = (uint64_t)(rem - (int64_t)comp * g.threads);
    uint64_t ctr = g.offset / 4 + (uint64_t)it;
    uint4 c = make_uint4((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)idx, (uint32_t)(idx >> 32));
    uint2 k = make_uint2((uint32_t)g.seed, (uint32_t)(g.seed >> 32));
    uint4 r = philox4x32_10(c, k);
    uint32_t x = comp == 0 ? r.x : comp == 1 ? r.y : comp == 2 ? r.z : r.w;
    // _curand_uniform: (0,1]
    float u = x * 2.3283064365386963e-10f + (2.3283064365386963e-10f / 2.0f);
    const float eps = 1.1920928955078125e-07f;  // numeric_limits<float>::epsilon()
    // at::log on device is the fast __logf (ATen/NumericUtils.h:150-160): lg2.approx * ln2
    float lg = (u >= 1.0f - eps / 2.0f) ? (-eps / 2.0f) : __logf(u);
    return -1.0f / 1.0f * lg;
}

// Generator offset and first q element of row `gi` (index inside the logical call) at step t.
// n_cand == 0, the global mapping: one torch.multinomial((N_total, V), 1) per step -> offset + t*inc, element gi*V.
// n_cand > 0, per-memory streams: the n_cand rows of memory column c = gi / n_cand are one torch.multinomial((n_cand, V), 1)
// per step, the columns' calls taken in order (max_len = col_steps calls per column) -> offset + (c*col_steps + t)*inc,
// element (gi mod n_cand)*V of that call's n_cand*V tensor (g.threads must be torch_rng_threads(n_cand*V)).
__host__ __device__ __forceinline__ int64_t torch_rng_row(RngGeom& g, uint64_t inc, int64_t n_cand, int64_t col_steps,
                                                          int64_t gi, int t, int V) {
    if (n_cand <= 0) {
        g.offset += (uint64_t)t * inc;
        return gi * V;
    }
    const int64_t c = gi / n_cand;
    g.offset += ((uint64_t)c * (uint64_t)col_steps + (uint64_t)t) * inc;
    return (gi - c * n_cand) * V;
}

}  // namespace mmt
