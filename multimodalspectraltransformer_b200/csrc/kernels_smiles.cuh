// Distinct SMILES per memory column on the device (mmt_distinct_smiles).
//
// A candidate's string is the byte concatenation of the itos entries of its ids before the first <EOS>
// (tensor_to_smiles, helper_functions_pl_v15_4.py:247-269).  Two candidates are the same string when their BYTES are
// equal: an itos may spell one string with different ids ("C","l" and "Cl").  A 64-bit FNV-1a hash of the bytes picks
// which candidates to compare; equality is always decided byte by byte.
//
//   smiles_dedup   one CTA per memory column: EOS length, byte length and hash of every candidate, then the first
//                  occurrence of each string through an open-addressing table of candidate indices (shared memory up
//                  to SMILES_SMEM_SLOTS slots, a global slice per column beyond), then multiplicities.
//   smiles_scan    one CTA: exclusive scans of the distinct flags and of their byte lengths (output slot and byte offset).
//   smiles_emit    one thread per candidate: a distinct string writes its metadata and its bytes contiguously.
#pragma once
#include "common.cuh"

namespace mmt {

constexpr int SMILES_SMEM_SLOTS = 8192;      // 32 KB of int: columns of up to 4,096 candidates keep the table in shared memory

struct SmilesParams {
    const int64_t* tokens;     // (T, N) ids
    int T; int64_t N; int k;   // k candidates per column, N = Bm * k
    int64_t eos;
    const uint8_t* tab_bytes;  // itos entries, UTF-8, concatenated
    const int2* tab;           // [n_tab] {byte start, byte length}, length < 0: the id has no itos entry
    int n_tab;
    int P;                     // table slots per column (power of two >= 2k)
    int* gtable;               // [Bm][P] when P > SMILES_SMEM_SLOTS, else unused
    int32_t* ntok;             // [N] ids before the first <EOS>
    int64_t* nbytes;           // [N] bytes of the string
    uint64_t* hash;            // [N]
    int32_t* slot;             // [N] table slot of the candidate's string
    int32_t* mult;             // [N] multiplicity, at the first occurrence
    int32_t* isd;              // [N] 1 at the first occurrence of a string
    int64_t* bad;              // {flag, id}: an id before <EOS> without itos entry
};

__device__ __forceinline__ int2 smiles_entry(const SmilesParams& p, int64_t id) {
    if (id < 0 || id >= p.n_tab) return make_int2(0, -1);
    return p.tab[id];
}

// byte equality of candidates a and b (same column), given equal hashes and byte lengths: two cursors over the
// itos entries of their ids (entries of invalid ids count as empty, as in smiles_dedup's byte count)
__device__ bool smiles_equal(const SmilesParams& p, int64_t a, int64_t b) {
    if (p.hash[a] != p.hash[b] || p.nbytes[a] != p.nbytes[b]) return false;
    int64_t left = p.nbytes[a];
    int ta = 0, tb = 0, na = 0, nb = 0;
    const uint8_t *sa = nullptr, *sb = nullptr;
    while (left > 0) {
        while (na == 0) { const int2 e = smiles_entry(p, p.tokens[(int64_t)ta++ * p.N + a]); sa = p.tab_bytes + e.x; na = max(e.y, 0); }
        while (nb == 0) { const int2 e = smiles_entry(p, p.tokens[(int64_t)tb++ * p.N + b]); sb = p.tab_bytes + e.x; nb = max(e.y, 0); }
        const int m = min(na, nb);
        for (int j = 0; j < m; ++j) if (sa[j] != sb[j]) return false;
        sa += m; sb += m; na -= m; nb -= m; left -= m;
    }
    return true;
}

__global__ void __launch_bounds__(1024) smiles_dedup(const __grid_constant__ SmilesParams p) {
    extern __shared__ int stab[];
    const int col = blockIdx.x;
    const int64_t base = (int64_t)col * p.k;
    int* tab = p.P <= SMILES_SMEM_SLOTS ? stab : p.gtable + (int64_t)col * p.P;
    for (int j = threadIdx.x; j < p.P; j += blockDim.x) tab[j] = -1;
    // lengths and hashes; ids are read time-major, consecutive candidates by consecutive threads
    for (int i = threadIdx.x; i < p.k; i += blockDim.x) {
        const int64_t n = base + i;
        uint64_t h = 0xcbf29ce484222325ull;
        int64_t nb = 0;
        int L = p.T;
        for (int t = 0; t < p.T; ++t) {
            const int64_t id = p.tokens[(int64_t)t * p.N + n];
            if (id == p.eos) { L = t; break; }
            const int2 e = smiles_entry(p, id);
            if (e.y < 0) { p.bad[1] = id; p.bad[0] = 1; continue; }
            for (int j = 0; j < e.y; ++j) h = (h ^ p.tab_bytes[e.x + j]) * 0x100000001b3ull;
            nb += e.y;
        }
        p.ntok[n] = L; p.nbytes[n] = nb; p.hash[n] = h; p.mult[n] = 0;
    }
    __syncthreads();
    // first occurrence: a slot is claimed by the first candidate of a string to reach it and then only ever holds
    // candidates of that string, so atomicMin leaves it at the string's lowest index
    const int mask = p.P - 1;
    for (int i = threadIdx.x; i < p.k; i += blockDim.x) {
        const int64_t n = base + i;
        const uint64_t h = p.hash[n];
        int s = (int)((h ^ (h >> 32)) & (uint64_t)mask);
        while (true) {
            const int cur = atomicCAS(&tab[s], -1, i);
            if (cur == -1) break;
            if (smiles_equal(p, base + cur, n)) { atomicMin(&tab[s], i); break; }
            s = (s + 1) & mask;
        }
        p.slot[n] = s;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < p.k; i += blockDim.x) {
        const int64_t n = base + i;
        const int first = tab[p.slot[n]];
        p.isd[n] = first == i;
        atomicAdd(&p.mult[base + first], 1);
    }
}

// didx = exclusive scan of isd, dbyte = exclusive scan of isd * nbytes; entry N holds the totals.  One CTA of 1024
// threads, tiles of 8 consecutive items per thread.
__global__ void __launch_bounds__(1024) smiles_scan(const int32_t* isd, const int64_t* nbytes, int64_t N, int64_t* didx, int64_t* dbyte) {
    constexpr int IT = 8;
    __shared__ int64_t wc[32], wb[32];
    __shared__ int64_t carry_c, carry_b;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) { carry_c = 0; carry_b = 0; }
    __syncthreads();
    for (int64_t t0 = 0; t0 < N; t0 += (int64_t)blockDim.x * IT) {
        const int64_t i0 = t0 + (int64_t)tid * IT;
        int64_t c = 0, b = 0;
        for (int j = 0; j < IT; ++j) if (i0 + j < N && isd[i0 + j]) { ++c; b += nbytes[i0 + j]; }
        int64_t ic = c, ib = b;          // inclusive warp scan
        for (int o = 1; o < 32; o <<= 1) {
            const int64_t uc = __shfl_up_sync(0xffffffffu, ic, o), ub = __shfl_up_sync(0xffffffffu, ib, o);
            if (lane >= o) { ic += uc; ib += ub; }
        }
        if (lane == 31) { wc[warp] = ic; wb[warp] = ib; }
        __syncthreads();
        if (warp == 0) {
            int64_t xc = lane < (int)(blockDim.x >> 5) ? wc[lane] : 0, xb = lane < (int)(blockDim.x >> 5) ? wb[lane] : 0;
            for (int o = 1; o < 32; o <<= 1) {
                const int64_t uc = __shfl_up_sync(0xffffffffu, xc, o), ub = __shfl_up_sync(0xffffffffu, xb, o);
                if (lane >= o) { xc += uc; xb += ub; }
            }
            wc[lane] = xc; wb[lane] = xb;   // inclusive over warps
        }
        __syncthreads();
        int64_t rc = carry_c + (warp ? wc[warp - 1] : 0) + ic - c;
        int64_t rb = carry_b + (warp ? wb[warp - 1] : 0) + ib - b;
        for (int j = 0; j < IT; ++j) {
            if (i0 + j >= N) break;
            didx[i0 + j] = rc; dbyte[i0 + j] = rb;
            if (isd[i0 + j]) { ++rc; rb += nbytes[i0 + j]; }
        }
        __syncthreads();
        if (tid == 0) { carry_c += wc[(blockDim.x >> 5) - 1]; carry_b += wb[(blockDim.x >> 5) - 1]; }
        __syncthreads();
    }
    if (tid == 0) { didx[N] = carry_c; dbyte[N] = carry_b; }
}

// Output, int64 unless noted (D = didx[N] distinct strings, Bm columns):
//   col_off [Bm+1]  strings of column b are [col_off[b], col_off[b+1])
//   first [D], count [D], ntok [D]   first candidate (index inside the column), multiplicity, ids before <EOS>
//   boff [D+1]      bytes of string d are [boff[d], boff[d+1]) of ...
//   bytes (uint8)   ... the UTF-8 strings, contiguous
__global__ void smiles_emit(const SmilesParams p, const int64_t* didx, const int64_t* dbyte, int64_t Bm, int64_t* out) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= p.N) return;
    const int64_t Dn = didx[p.N];
    int64_t* col_off = out;
    int64_t* first = col_off + Bm + 1;
    int64_t* count = first + Dn;
    int64_t* ntok = count + Dn;
    int64_t* boff = ntok + Dn;
    uint8_t* bytes = reinterpret_cast<uint8_t*>(boff + Dn + 1);
    const int64_t col = n / p.k;
    if (n == col * p.k) col_off[col] = didx[n];
    if (n == 0) { col_off[Bm] = Dn; boff[Dn] = dbyte[p.N]; }
    if (!p.isd[n]) return;
    const int64_t d = didx[n];
    first[d] = n - col * p.k; count[d] = p.mult[n]; ntok[d] = p.ntok[n]; boff[d] = dbyte[n];
    uint8_t* o = bytes + dbyte[n];
    for (int t = 0; t < p.ntok[n]; ++t) {
        const int2 e = smiles_entry(p, p.tokens[(int64_t)t * p.N + n]);
        for (int j = 0; j < e.y; ++j) *o++ = p.tab_bytes[e.x + j];
    }
}

}  // namespace mmt
