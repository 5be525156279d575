// grmkm_patterns.cuh -- the distinct presence patterns of the resident result (grmkm_patterns): columns grouped by exact
// equality of their W words and of a per-column class byte, numbered in the order of their first column.
//
//   k_pat_hash    fp[j] = a 64-bit fingerprint of column j's words and class, read at the matrix pitch (a warp covers
//                 32 consecutive columns: every word row is one coalesced load), truncated to GRMKM_PATTERN_HASH_BITS.
//   k_pat_insert  one round of grouping: every active column finds its fingerprint's slot in an open-addressing table
//                 (linear probing, CAS on the key) and leaves its index there with atomicMin: the slot's head is the
//                 least active column of that fingerprint, whatever the order of the atomics.
//   k_pat_verify  every active column compares its words and class with its slot's head.  Equal: it is a member of
//                 that head (the head is a member of itself).  Different (a fingerprint collision): it goes to the next
//                 round, which builds a fresh table without the heads settled so far.  Every occupied slot settles its
//                 head, so each round settles at least one column and the rounds end.
//   k_pat_assign  after an exclusive scan of "is a head" in column order (pid): pattern_of[j] = pid[head_of[j]], the
//                 head column of every pattern, its multiplicity, and the values (column indices) of the stable sort by
//                 pattern that lists the members of every pattern in ascending order.
//
// The columns of one pattern share their fingerprint, so they meet in every round until the round in which their least
// column is a head; all of them join it then.  The result is therefore the exact grouping, numbered by first column,
// for any grid, any order of the atomics and any fingerprint width.
#pragma once
#include <cstdint>

namespace grmkm {

constexpr unsigned long long kPatEmpty = ~0ULL;      // free table slot; no fingerprint takes this value

__device__ __forceinline__ unsigned long long pat_mix(unsigned long long x) {      // murmur3 fmix64
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}

__global__ void __launch_bounds__(256)
k_pat_hash(const unsigned long long* __restrict__ matrix, unsigned long long pitch, uint32_t W, uint32_t U,
           const uint8_t* __restrict__ cls /* U bytes or null */, uint32_t bits, unsigned long long* __restrict__ fp) {
    for (unsigned long long j = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j < U;
         j += (unsigned long long)gridDim.x * blockDim.x) {
        unsigned long long h = pat_mix(0x9E3779B97F4A7C15ULL + (cls ? cls[j] : 0u));
        for (uint32_t w = 0; w < W; ++w) h = pat_mix(h ^ matrix[(unsigned long long)w * pitch + j]) + 0x9E3779B97F4A7C15ULL;
        if (bits < 64) h &= (1ULL << bits) - 1;
        fp[j] = h == kPatEmpty ? h - 1 : h;
    }
}

// act: the active columns of the round (null: all of 0..n-1); slot_of[i]: the slot of act[i]
__global__ void __launch_bounds__(256)
k_pat_insert(const uint32_t* __restrict__ act, uint32_t n, const unsigned long long* __restrict__ fp,
             unsigned long long* __restrict__ tkey, uint32_t* __restrict__ thead, unsigned long long mask,
             uint32_t* __restrict__ slot_of) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t j = act ? act[i] : (uint32_t)i;
        const unsigned long long h = fp[j];
        unsigned long long s = pat_mix(h) & mask;
        for (;;) {      // the table has at least twice as many slots as active columns: a free slot is always found
            unsigned long long k = tkey[s];
            if (k == kPatEmpty) {
                k = atomicCAS(tkey + s, kPatEmpty, h);
                if (k == kPatEmpty) k = h;
            }
            if (k == h) break;
            s = (s + 1) & mask;
        }
        atomicMin(thead + s, j);
        slot_of[i] = (uint32_t)s;
    }
}

__global__ void __launch_bounds__(256)
k_pat_verify(const unsigned long long* __restrict__ matrix, unsigned long long pitch, uint32_t W,
             const uint8_t* __restrict__ cls, const uint32_t* __restrict__ act, uint32_t n,
             const uint32_t* __restrict__ slot_of, const uint32_t* __restrict__ thead, uint32_t* __restrict__ head_of,
             uint32_t* __restrict__ next, unsigned int* __restrict__ n_next) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t j = act ? act[i] : (uint32_t)i;
        const uint32_t h = thead[slot_of[i]];
        bool same = !cls || cls[j] == cls[h];
        for (uint32_t w = 0; same && w < W && h != j; ++w)
            same = matrix[(unsigned long long)w * pitch + j] == matrix[(unsigned long long)w * pitch + h];
        if (same) head_of[j] = h;
        else next[atomicAdd(n_next, 1u)] = j;
    }
}

// flag[j] = 1 iff column j heads its pattern (flag[U] = 0: the scan's last entry is P)
__global__ void __launch_bounds__(256)
k_pat_flags(const uint32_t* __restrict__ head_of, uint32_t U, uint32_t* __restrict__ flag) {
    for (unsigned long long j = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j <= U;
         j += (unsigned long long)gridDim.x * blockDim.x)
        flag[j] = j < U && head_of[j] == (uint32_t)j;
}

// mult must be zero on entry
__global__ void __launch_bounds__(256)
k_pat_assign(const uint32_t* __restrict__ head_of, const uint32_t* __restrict__ pid, uint32_t U,
             uint32_t* __restrict__ pattern_of, uint32_t* __restrict__ col, unsigned long long* __restrict__ heads,
             uint32_t* __restrict__ mult) {
    for (unsigned long long j = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; j < U;
         j += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t h = head_of[j], p = pid[h];
        pattern_of[j] = p;
        col[j] = (uint32_t)j;
        if (h == (uint32_t)j) heads[p] = j;
        atomicAdd(mult + p, 1u);
    }
}

}  // namespace grmkm
