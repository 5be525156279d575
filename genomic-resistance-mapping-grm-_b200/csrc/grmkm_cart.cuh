// grmkm_cart.cuh -- CART decision trees (kover learning/learners/cart.py, `kover learn tree`, gini criterion) on the
// resident matrix.  A node splits on k-mer column j < U: the examples holding the k-mer go to the present child, the
// others to the absent child.  Trees grow breadth-first; every level of a whole batch of trees is one pass over the
// matrix per chunk of open nodes:
//
//   k_cart_scan   every column's words are read once and ANDed and popcounted against the P and N masks of every open
//                 node of the chunk (shared memory); every admissible split (both children non-empty, k-mer not
//                 blacklisted) gets its score (A_l B_l)/S_l + (A_r B_r)/S_r, and every CTA keeps each node's least score
//                 as ~scm_key(score) (largest key = least score; scores are >= +0.0, so 0 stays "no split").  Per node:
//                 the CTA's best goes to tile_best[f][cta], the global best to best[slot] (atomicMax).  No per-column
//                 array is written.
//   k_cart_ties   the targeted second pass, twice: only the CTAs holding a node's best revisit their columns.  The count
//                 pass writes the node's number of ties in the CTA's columns to tile_cnt[f][cta] and adds it to
//                 total[slot].  The append pass appends (slot << 32) | j for every tie of a CTA only if the CTAs before
//                 it hold fewer than the node's `need` ties: each CTA covers one contiguous column range, so the `need`
//                 smallest members of T are always in the list, and the list of a node holds fewer than
//                 need + (columns of one CTA) entries however large T is.  The list is complete for what the host
//                 keeps or its counter says by how much it overflowed (the host grows it and redoes the level).
//                 WEIGHTED (a pattern matrix, grmkm_patterns): total[slot] adds every tie column's multiplicity mult[j],
//                 so it counts k-mers; tile_cnt, and with it the append cap, still counts columns (patterns).
//   k_cart_gather pL, nL of the chosen rule of every split node (all of T share the score, not the counts).
//   k_cart_split  P & col, P & ~col, N & col, N & ~col of every split node into the masks of its open children.
//
// Masks: masks[slot][0..1][W] = P, N of the open nodes of the level (genome g at bit 63 - g % 64 of word g / 64).  The
// scan and both tie passes use the same grid and the same column ranges, so tile_best / tile_cnt index the same columns
// in all three; the results do not depend on the grid.
#pragma once
#include <cstdint>

#include "grmkm_scm.cuh"

namespace grmkm {

struct CartNodeArg {
    double w_pos, w_neg;      // class importances
    unsigned long long need;  // max(1, equiv_cap): the node's smallest tie members the list must hold
    uint32_t slot;            // the node's position among the open nodes of the level: masks / best / total
    uint32_t n_pos, n_neg;    // |P|, |N|
    uint32_t pad;
};

struct CartSplit {
    uint32_t src;             // slot of the split node
    uint32_t j;               // its k-mer column
    uint32_t dst_present;     // slot of the present child in the next level's masks, UINT32_MAX: not open
    uint32_t dst_absent;      // the same for the absent child
};

// half the weighted Gini impurity of a child holding a positive and b negative examples (a + b > 0):
// A = w_pos a, B = w_neg b, (A B) / (A + B), every operation correctly rounded in this order (numpy's (A*B)/S)
__device__ __forceinline__ double cart_term(uint32_t a, uint32_t b, double w_pos, double w_neg) {
    const double A = __dmul_rn(w_pos, (double)a), B = __dmul_rn(w_neg, (double)b);
    return __ddiv_rn(__dmul_rn(A, B), __dadd_rn(A, B));
}

// key of split (pl, nl) of a node of |P| = np, |N| = nn: 0 if inadmissible, else larger for a smaller score
__device__ __forceinline__ unsigned long long cart_key(uint32_t pl, uint32_t nl, uint32_t np, uint32_t nn, double w_pos,
                                                       double w_neg) {
    const uint32_t pr = np - pl, nr = nn - nl;
    if (!(pl | nl) || !(pr | nr)) return 0ULL;
    return ~scm_key(__dadd_rn(cart_term(pl, nl, w_pos, w_neg), cart_term(pr, nr, w_pos, w_neg)));
}

// the SCM's shared-memory layout (P, N, per-warp bests, p -> w_pos, |P|, |N|) plus w_neg[n]
__host__ __device__ inline size_t cart_smem_bytes(uint32_t n, uint32_t W) { return scm_smem_bytes(n, W) + (size_t)n * 8; }

__device__ __forceinline__ double* cart_w_neg(const ScmShared& s, uint32_t n) { return (double*)(s.n_neg + n); }

__device__ __forceinline__ void cart_load_chunk(const ScmShared& s, const CartNodeArg* __restrict__ args, uint32_t n,
                                                uint32_t W, const unsigned long long* __restrict__ masks) {
    for (uint32_t i = threadIdx.x; i < n * W; i += blockDim.x) {
        const uint32_t f = i / W, w = i - f * W;
        const unsigned long long* m = masks + (size_t)args[f].slot * 2 * W;
        s.P[i] = m[w];
        s.N[i] = m[W + w];
    }
    double* w_neg = cart_w_neg(s, n);
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        s.p[f] = args[f].w_pos;
        w_neg[f] = args[f].w_neg;
        s.n_pos[f] = args[f].n_pos;
        s.n_neg[f] = args[f].n_neg;
    }
}

// CTA b covers tiles [b tpc, (b + 1) tpc) of 256 columns
template <bool CACHED>
__global__ void __launch_bounds__(kScmThreads)
k_cart_scan(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
            const uint32_t* __restrict__ blacklist /* U bits */, const CartNodeArg* __restrict__ args, uint32_t n,
            const unsigned long long* __restrict__ masks, unsigned long long tpc,
            unsigned long long* __restrict__ best /* [slots] */, unsigned long long* __restrict__ tile_best /* [n][grid] */) {
    extern __shared__ unsigned long long scm_sm[];
    const ScmShared s = scm_shared(scm_sm, n, W);
    const double* w_neg = cart_w_neg(s, n);
    cart_load_chunk(s, args, n, W, masks);
    for (uint32_t i = threadIdx.x; i < n * kScmWarps; i += blockDim.x) s.aux[i] = 0;
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const unsigned long long n_tiles = (U + kScmThreads - 1) / kScmThreads;
    const unsigned long long t0 = blockIdx.x * tpc, t1 = t0 + tpc < n_tiles ? t0 + tpc : n_tiles;
    unsigned long long col[CACHED ? kScmCachedWords : 1];
    for (unsigned long long t = t0; t < t1; ++t) {
        const unsigned long long j = t * kScmThreads + threadIdx.x;
        const bool valid = j < U;
        scm_load_col<CACHED>(col, matrix, pitch, W, j, valid);
        const bool ok = valid && !scm_blacklisted(blacklist, j);
        for (uint32_t f = 0; f < n; ++f) {
            unsigned long long k = 0;
            if (ok) {
                uint32_t pl, nl;
                scm_counts<CACHED>(s, f, W, col, matrix, pitch, j, pl, nl);
                k = cart_key(pl, nl, s.n_pos[f], s.n_neg[f], s.p[f], w_neg[f]);
            }
            k = warp_max_u64(k);
            if (lane == 0 && k > s.aux[f * kScmWarps + warp]) s.aux[f * kScmWarps + warp] = k;
        }
    }
    __syncthreads();
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        unsigned long long v = 0;
        for (uint32_t w = 0; w < kScmWarps; ++w) v = v > s.aux[f * kScmWarps + w] ? v : s.aux[f * kScmWarps + w];
        tile_best[(size_t)f * gridDim.x + blockIdx.x] = v;
        if (v) atomicMax(best + args[f].slot, v);
    }
}

// append = 0: the count pass (tile_cnt, total); append = 1: the append pass (list, count).  mult: WEIGHTED only, the
// columns' multiplicities
template <bool CACHED, bool WEIGHTED = false>
__global__ void __launch_bounds__(kScmThreads)
k_cart_ties(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
            const uint32_t* __restrict__ blacklist, const CartNodeArg* __restrict__ args, uint32_t n,
            const unsigned long long* __restrict__ masks, unsigned long long tpc, const unsigned long long* __restrict__ best,
            const unsigned long long* __restrict__ tile_best, uint32_t* __restrict__ tile_cnt /* [n][grid] */,
            unsigned long long* __restrict__ total /* [slots] */, int append, unsigned long long* __restrict__ list,
            unsigned long long* __restrict__ count, unsigned long long cap, const uint32_t* __restrict__ mult = nullptr) {
    static_assert(kScmWarps >= 2, "the tie passes keep two words per node in the per-warp area");
    extern __shared__ unsigned long long scm_sm[];
    const ScmShared s = scm_shared(scm_sm, n, W);
    unsigned long long* key = s.aux;         // key[f]: the node's best if this CTA holds it (and, appending, may append)
    unsigned long long* cnt = s.aux + n;     // cnt[f]: ties of the node in this CTA's columns / ties before this CTA
    __shared__ int any;
    if (threadIdx.x == 0) any = 0;
    __syncthreads();
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        const unsigned long long b = best[args[f].slot];
        const bool mine = b && tile_best[(size_t)f * gridDim.x + blockIdx.x] == b;
        key[f] = mine ? b : 0ULL;
        cnt[f] = 0;
        if (mine) any = 1;
        else if (!append) tile_cnt[(size_t)f * gridDim.x + blockIdx.x] = 0;
    }
    __syncthreads();
    if (!any) return;
    if (append) {
        // ties of the node in the columns of the CTAs before this one; at `need` or more this CTA adds nothing
        for (uint32_t f = 0; f < n; ++f) {
            if (!key[f]) continue;
            unsigned long long v = 0;
            for (uint32_t b = threadIdx.x; b < blockIdx.x; b += blockDim.x) v += tile_cnt[(size_t)f * gridDim.x + b];
            v = __reduce_add_sync(0xffffffffu, (uint32_t)v);      // < 2^31: at most U ties in all
            if ((threadIdx.x & 31u) == 0 && v) atomicAdd(cnt + f, v);
        }
        __syncthreads();
        for (uint32_t f = threadIdx.x; f < n; f += blockDim.x)
            if (key[f] && cnt[f] >= args[f].need) key[f] = 0;
        __syncthreads();
    }
    cart_load_chunk(s, args, n, W, masks);
    __syncthreads();
    const double* w_neg = cart_w_neg(s, n);
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned long long n_tiles = (U + kScmThreads - 1) / kScmThreads;
    const unsigned long long t0 = blockIdx.x * tpc, t1 = t0 + tpc < n_tiles ? t0 + tpc : n_tiles;
    unsigned long long col[CACHED ? kScmCachedWords : 1];
    for (unsigned long long t = t0; t < t1; ++t) {
        const unsigned long long j = t * kScmThreads + threadIdx.x;
        const bool valid = j < U;
        scm_load_col<CACHED>(col, matrix, pitch, W, j, valid);
        const bool ok = valid && !scm_blacklisted(blacklist, j);
        for (uint32_t f = 0; f < n; ++f) {
            const unsigned long long b = key[f];
            if (!b) continue;
            bool tie = false;
            if (ok) {
                uint32_t pl, nl;
                scm_counts<CACHED>(s, f, W, col, matrix, pitch, j, pl, nl);
                tie = cart_key(pl, nl, s.n_pos[f], s.n_neg[f], s.p[f], w_neg[f]) == b;
            }
            // one atomic per warp: key[f] is the same in the whole CTA, so every lane reaches the ballot
            const uint32_t m = __ballot_sync(0xffffffffu, tie);
            if (!m) continue;
            if (append) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(count, (unsigned long long)__popc(m));
                base = __shfl_sync(0xffffffffu, base, 0);
                const unsigned long long i = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
                if (tie && i < cap) list[i] = ((unsigned long long)args[f].slot << 32) | j;
            } else {
                if (lane == 0) atomicAdd(cnt + f, (unsigned long long)__popc(m));
                if (WEIGHTED && tie) atomicAdd(total + args[f].slot, (unsigned long long)mult[j]);
            }
        }
    }
    if (append) return;
    __syncthreads();
    for (uint32_t f = threadIdx.x; f < n; f += blockDim.x) {
        if (!key[f]) continue;
        tile_cnt[(size_t)f * gridDim.x + blockIdx.x] = (uint32_t)cnt[f];
        if (!WEIGHTED && cnt[f]) atomicAdd(total + args[f].slot, cnt[f]);
    }
}

// one warp per split node: stats[2 i], stats[2 i + 1] = popcounts of column sp[i].j under its P and N
__global__ void __launch_bounds__(256)
k_cart_gather(const unsigned long long* __restrict__ matrix, unsigned long long pitch, uint32_t W,
              const unsigned long long* __restrict__ masks, const CartSplit* __restrict__ sp, uint32_t n,
              uint32_t* __restrict__ stats) {
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += (gridDim.x * blockDim.x) >> 5) {
        const unsigned long long* P = masks + (size_t)sp[i].src * 2 * W;
        uint32_t pl = 0, nl = 0;
        for (uint32_t w = lane; w < W; w += 32) {
            const unsigned long long x = matrix[(unsigned long long)w * pitch + sp[i].j];
            pl += (uint32_t)__popcll(x & P[w]);
            nl += (uint32_t)__popcll(x & P[W + w]);
        }
        pl = __reduce_add_sync(0xffffffffu, pl);
        nl = __reduce_add_sync(0xffffffffu, nl);
        if (lane == 0) { stats[2 * i] = pl; stats[2 * i + 1] = nl; }
    }
}

// the masks of the open children of every split node: present = P & col, N & col; absent = P & ~col, N & ~col
__global__ void __launch_bounds__(256)
k_cart_split(const unsigned long long* __restrict__ matrix, unsigned long long pitch, uint32_t W,
             const unsigned long long* __restrict__ masks, const CartSplit* __restrict__ sp, uint32_t n,
             unsigned long long* __restrict__ next) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < (unsigned long long)n * W;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t k = (uint32_t)(i / W), w = (uint32_t)(i - (unsigned long long)k * W);
        const CartSplit e = sp[k];
        const unsigned long long x = matrix[(unsigned long long)w * pitch + e.j];
        const unsigned long long P = masks[(size_t)e.src * 2 * W + w], N = masks[(size_t)e.src * 2 * W + W + w];
        if (e.dst_present != UINT32_MAX) {
            next[(size_t)e.dst_present * 2 * W + w] = P & x;
            next[(size_t)e.dst_present * 2 * W + W + w] = N & x;
        }
        if (e.dst_absent != UINT32_MAX) {
            next[(size_t)e.dst_absent * 2 * W + w] = P & ~x;
            next[(size_t)e.dst_absent * 2 * W + W + w] = N & ~x;
        }
    }
}

}  // namespace grmkm
