// grmkm_scm.cuh -- the Set Covering Machine's greedy step on the resident matrix (kover learning/learners/scm.py, the
// loop around KmerRuleClassifications.sum_rows, scm.py:238-288).  Rule r < U is "k-mer r present", rule U + r its
// absence twin.  A batch of fits (model type x p x fold) advances one rule per step:
//
//   k_scm_scan    one pass over the matrix per chunk of fits: every column's words are ANDed and popcounted against the
//                 P and N masks of every fit of the chunk (shared memory), both rules of the column get their utility
//                 u = c - p e, and every CTA keeps each fit's best utility (as an order-preserving 64-bit key).  Per fit:
//                 the CTA's best goes to tile_best[f][cta], the global best to best[fit] (atomicMax).  No per-rule array
//                 of counts or utilities is ever written.
//   k_scm_ties    the targeted second pass: a CTA revisits its columns only for the fits whose best it holds, and appends
//                 every rule with u == u* that changes something to one list ((fit << 32) | rule).  The list is complete or
//                 its counter says by how much it overflowed (the host grows it and reruns the pass).
//   k_scm_gather  per listed rule: its errors, covers and Kover's risk tiebreaker, by gathering its column.
//   k_scm_update  P and N of every fit that took a rule keep the examples on which the rule outputs 1.
//
// Masks: masks[fit][0..3][W] = P, N, P0, N0 (genome g at bit 63 - g % 64 of word g / 64).  The two passes use the
// same grid, so tile_best indexes the same columns in both; the results do not depend on the grid.
#pragma once
#include <cstdint>

namespace grmkm {

constexpr uint32_t kScmThreads = 256;
constexpr uint32_t kScmWarps = kScmThreads / 32;
constexpr uint32_t kScmCachedWords = 8;      // matrices of up to 8 word rows (512 genomes) keep a column in registers

struct ScmFitArg {
    double p;
    uint32_t fit;         // index into masks / best
    uint32_t n_pos, n_neg;  // |P|, |N|
    uint32_t pad;
};

// (double)c - p * (double)e with the product rounded, then the difference (numpy's order; never an FMA)
__device__ __forceinline__ double scm_utility(uint32_t c, uint32_t e, double p) {
    return __dsub_rn((double)c, __dmul_rn(p, (double)e));
}

// order-preserving key of a double (no NaN, no -0.0 here); 0 = "no rule"
__device__ __forceinline__ unsigned long long scm_key(double u) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(u);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long k) {
    const uint32_t hi = (uint32_t)(k >> 32), mh = __reduce_max_sync(0xffffffffu, hi);
    const uint32_t m = __ballot_sync(0xffffffffu, hi == mh);
    uint32_t ml = 0;
    if (hi == mh) ml = __reduce_max_sync(m, (uint32_t)k);
    ml = __shfl_sync(0xffffffffu, ml, __ffs(m) - 1);
    return ((unsigned long long)mh << 32) | ml;
}

__device__ __forceinline__ bool scm_blacklisted(const uint32_t* __restrict__ bl, unsigned long long r) {
    return (bl[r >> 5] >> (r & 31)) & 1u;
}

// shared memory of both passes: P[n][W], N[n][W], per-warp bests (scan) or per-fit flags (ties), p, |P|, |N|
__host__ __device__ inline size_t scm_smem_bytes(uint32_t n, uint32_t W) {
    return (size_t)n * (2 * (size_t)W + kScmWarps) * 8 + (size_t)n * (8 + 4 + 4);
}

struct ScmShared {
    unsigned long long *P, *N, *aux;
    double* p;
    uint32_t *n_pos, *n_neg;
};

__device__ __forceinline__ ScmShared scm_shared(unsigned long long* sm, uint32_t n, uint32_t W) {
    ScmShared s;
    s.P = sm;
    s.N = sm + (size_t)n * W;
    s.aux = sm + (size_t)2 * n * W;
    s.p = (double*)(s.aux + (size_t)n * kScmWarps);
    s.n_pos = (uint32_t*)(s.p + n);
    s.n_neg = s.n_pos + n;
    return s;
}

__device__ __forceinline__ void scm_load_chunk(const ScmShared& s, const ScmFitArg* __restrict__ args, uint32_t n, uint32_t W,
                                               const unsigned long long* __restrict__ masks) {
    for (uint32_t i = threadIdx.x; i < n * W; i += blockDim.x) {
        const uint32_t f = i / W, w = i - f * W;
        const unsigned long long* m = masks + (size_t)args[f].fit * 4 * W;
        s.P[i] = m[w];
        s.N[i] = m[W + w];
    }
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        s.p[f] = args[f].p;
        s.n_pos[f] = args[f].n_pos;
        s.n_neg[f] = args[f].n_neg;
    }
}

// popcounts of column j under fit f's P and N
template <bool CACHED>
__device__ __forceinline__ void scm_counts(const ScmShared& s, uint32_t f, uint32_t W, const unsigned long long* col,
                                           const unsigned long long* __restrict__ matrix, unsigned long long pitch,
                                           unsigned long long j, uint32_t& pp, uint32_t& pn) {
    const unsigned long long* P = s.P + (size_t)f * W;
    const unsigned long long* N = s.N + (size_t)f * W;
    pp = 0; pn = 0;
    if (CACHED) {
#pragma unroll
        for (uint32_t w = 0; w < kScmCachedWords; ++w)
            if (w < W) { pp += (uint32_t)__popcll(col[w] & P[w]); pn += (uint32_t)__popcll(col[w] & N[w]); }
    } else {
        for (uint32_t w = 0; w < W; ++w) {
            const unsigned long long x = __ldg(matrix + (unsigned long long)w * pitch + j);
            pp += (uint32_t)__popcll(x & P[w]);
            pn += (uint32_t)__popcll(x & N[w]);
        }
    }
}

template <bool CACHED>
__device__ __forceinline__ void scm_load_col(unsigned long long* col, const unsigned long long* __restrict__ matrix,
                                             unsigned long long pitch, uint32_t W, unsigned long long j, bool valid) {
    if (CACHED) {
#pragma unroll
        for (uint32_t w = 0; w < kScmCachedWords; ++w)
            col[w] = (valid && w < W) ? __ldcs(matrix + (unsigned long long)w * pitch + j) : 0ULL;
    }
}

template <bool CACHED>
__global__ void __launch_bounds__(kScmThreads)
k_scm_scan(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
           const uint32_t* __restrict__ blacklist /* 2U bits */, const ScmFitArg* __restrict__ args, uint32_t n,
           const unsigned long long* __restrict__ masks, unsigned long long* __restrict__ best /* [fits] */,
           unsigned long long* __restrict__ tile_best /* [n][gridDim.x] */) {
    extern __shared__ unsigned long long scm_sm[];
    const ScmShared s = scm_shared(scm_sm, n, W);
    scm_load_chunk(s, args, n, W, masks);
    for (uint32_t i = threadIdx.x; i < n * kScmWarps; i += blockDim.x) s.aux[i] = 0;
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const unsigned long long n_tiles = (U + kScmThreads - 1) / kScmThreads;
    unsigned long long col[CACHED ? kScmCachedWords : 1];
    for (unsigned long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const unsigned long long j = t * kScmThreads + threadIdx.x;
        const bool valid = j < U;
        scm_load_col<CACHED>(col, matrix, pitch, W, j, valid);
        const bool ok_p = valid && !scm_blacklisted(blacklist, j), ok_a = valid && !scm_blacklisted(blacklist, U + j);
        for (uint32_t f = 0; f < n; ++f) {
            uint32_t pp = 0, pn = 0;
            if (ok_p || ok_a) scm_counts<CACHED>(s, f, W, col, matrix, pitch, j, pp, pn);
            const double p = s.p[f];
            const unsigned long long kp = ok_p ? scm_key(scm_utility(s.n_neg[f] - pn, s.n_pos[f] - pp, p)) : 0ULL;
            const unsigned long long ka = ok_a ? scm_key(scm_utility(pn, pp, p)) : 0ULL;
            const unsigned long long k = warp_max_u64(kp > ka ? kp : ka);
            if (lane == 0 && k > s.aux[f * kScmWarps + warp]) s.aux[f * kScmWarps + warp] = k;
        }
    }
    __syncthreads();
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        unsigned long long v = 0;
        for (uint32_t w = 0; w < kScmWarps; ++w) v = v > s.aux[f * kScmWarps + w] ? v : s.aux[f * kScmWarps + w];
        tile_best[(size_t)f * gridDim.x + blockIdx.x] = v;
        if (v) atomicMax(best + args[f].fit, v);
    }
}

template <bool CACHED>
__global__ void __launch_bounds__(kScmThreads)
k_scm_ties(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
           const uint32_t* __restrict__ blacklist, const ScmFitArg* __restrict__ args, uint32_t n,
           const unsigned long long* __restrict__ masks, const unsigned long long* __restrict__ best,
           const unsigned long long* __restrict__ tile_best, unsigned long long* __restrict__ list,
           unsigned long long* __restrict__ count, unsigned long long cap) {
    extern __shared__ unsigned long long scm_sm[];
    const ScmShared s = scm_shared(scm_sm, n, W);
    __shared__ int any;
    if (threadIdx.x == 0) any = 0;
    __syncthreads();
    // s.aux[f] = u* of fit f if this CTA holds one of its best rules, else 0
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        const unsigned long long b = best[args[f].fit];
        const bool mine = b && tile_best[(size_t)f * gridDim.x + blockIdx.x] == b;
        s.aux[f] = mine ? b : 0ULL;
        if (mine) any = 1;
    }
    __syncthreads();
    if (!any) return;
    scm_load_chunk(s, args, n, W, masks);
    __syncthreads();
    const unsigned long long n_tiles = (U + kScmThreads - 1) / kScmThreads;
    unsigned long long col[CACHED ? kScmCachedWords : 1];
    for (unsigned long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        const unsigned long long j = t * kScmThreads + threadIdx.x;
        const bool valid = j < U;
        scm_load_col<CACHED>(col, matrix, pitch, W, j, valid);
        const bool ok_p = valid && !scm_blacklisted(blacklist, j), ok_a = valid && !scm_blacklisted(blacklist, U + j);
        if (!ok_p && !ok_a) continue;
        for (uint32_t f = 0; f < n; ++f) {
            const unsigned long long b = s.aux[f];
            if (!b) continue;
            uint32_t pp, pn;
            scm_counts<CACHED>(s, f, W, col, matrix, pitch, j, pp, pn);
            const double p = s.p[f];
            const uint32_t ep = s.n_pos[f] - pp, cp = s.n_neg[f] - pn;
            const unsigned long long fit = (unsigned long long)args[f].fit << 32;
            // a rule that changes nothing (no error, no cover) is never chosen
            if (ok_p && (ep | cp) && scm_key(scm_utility(cp, ep, p)) == b) {
                const unsigned long long i = atomicAdd(count, 1ULL);
                if (i < cap) list[i] = fit | j;
            }
            if (ok_a && (pp | pn) && scm_key(scm_utility(pn, pp, p)) == b) {
                const unsigned long long i = atomicAdd(count, 1ULL);
                if (i < cap) list[i] = fit | (U + j);
            }
        }
    }
}

// stats[3 i .. 3 i + 2] = errors on P, covers of N, risk (errors on P0 + N0 examples it outputs 1 on) of list entry i
__global__ void __launch_bounds__(256)
k_scm_gather(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
             const unsigned long long* __restrict__ masks, const unsigned long long* __restrict__ list, unsigned long long n,
             uint32_t* __restrict__ stats) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long e = list[i], fit = e >> 32, r = e & 0xffffffffULL;
        const bool absent = r >= U;
        const unsigned long long j = absent ? r - U : r;
        const unsigned long long* m = masks + fit * 4 * W;
        uint32_t err = 0, cov = 0, risk = 0;
        for (uint32_t w = 0; w < W; ++w) {
            const unsigned long long x = matrix[(unsigned long long)w * pitch + j], out = absent ? ~x : x;
            err += (uint32_t)__popcll(m[w] & ~out);
            cov += (uint32_t)__popcll(m[W + w] & ~out);
            risk += (uint32_t)__popcll(m[2 * W + w] & ~out) + (uint32_t)__popcll(m[3 * W + w] & out);
        }
        stats[3 * i] = err; stats[3 * i + 1] = cov; stats[3 * i + 2] = risk;
    }
}

// sel[i] = (fit << 32) | rule: P and N of the fit keep the examples the rule outputs 1 on
__global__ void __launch_bounds__(256)
k_scm_update(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
             const unsigned long long* __restrict__ sel, uint32_t n, unsigned long long* __restrict__ masks) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n * W; i += gridDim.x * blockDim.x) {
        const uint32_t k = i / W, w = i - k * W;
        const unsigned long long e = sel[k], fit = e >> 32, r = e & 0xffffffffULL;
        const bool absent = r >= U;
        const unsigned long long x = matrix[(unsigned long long)w * pitch + (absent ? r - U : r)], out = absent ? ~x : x;
        masks[fit * 4 * W + w] &= out;
        masks[fit * 4 * W + W + w] &= out;
    }
}

}  // namespace grmkm
