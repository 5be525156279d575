// grmkm_query.cuh -- which genomes hold which k-mers of a query set, straight from the packed stream (grmkm_query).
//
// The front end of a build (staging, k_first_header, k_tile_tickets, k_pack) turns the text into the packed stream;
// instead of unit bounds and the unit scatter, one scan then looks every valid k-mer window up in an open-addressing
// table of the query's distinct canonical k-mers and records a hit for the window's genome row.  No dedupe, expansion
// or aggregate: the work is one read of the packed stream, and the output is the (word rows x query) bit plane.
//
//   k_query_scan    packed stream -> hits: presence bits (min_abundance 1) or per-row u32 counters (min_abundance > 1)
//   k_query_gather  plane or counters -> the caller's column order (a counter becomes a bit when it reaches
//                   min_abundance), one word row of the range after the other
#pragma once
#include "grmkm_units.cuh"

namespace grmkm {

constexpr int kQsThreads = 256;
// small query sets: the table's keys sit in every CTA's shared memory (slots = a power of two >= 2 Qd, so 4096 keys
// take at most 8192 slots = 64 KB); larger sets probe the table in global memory (L2-resident up to several million keys)
constexpr uint32_t kQuerySmemKeys = 4096;

// Home slot of a key: the top bits of fmix64(k-mer), not of the column-order hash k-mer * kHashMul.  A query set is
// often a contiguous stretch of a build's columns (ascending kHashMul product): under that hash its keys would all
// have their home slots in one stretch of the table and form one cluster that every probe landing there walks (the
// first 10^6 columns of the C2-shape build, queried so, took minutes on a B200).  fmix64 scatters them whatever their
// column order.

struct QueryScanParams {
    const unsigned long long* codes;     // packed stream of the batch: entry j of group g at bits 2j of codes[g]
    const uint32_t* valid;               // bit j of valid[g]: entry j is a base
    const uint64_t* scalars;             // S_STREAM_LEN
    const uint64_t* fss;                 // [n_files + 1] first stream entry of every file of the batch
    const FileDesc* files;               // .row = genome row - row0
    uint32_t n_files;
    uint32_t k;
    const unsigned long long* keys;      // [1 << slot_bits] canonical k-mers, kEmptyKey = free slot
    const uint32_t* idx;                 // [1 << slot_bits] slot -> index of its key
    uint32_t slot_bits;
    uint32_t row0;                       // first genome row of the range
    uint64_t qd;                         // distinct keys = plane columns
    unsigned long long* plane;           // presence: [word row - row0 / 64][qd]
    uint32_t* counts;                    // counters: [row - row0][qd]
    unsigned long long* totals;          // [0] valid windows, [1] hits
};

// One thread = one group of 32 stream entries (the windows ending in it), grid-stride.  The window ending at entry e
// is valid iff entries e - k + 1 .. e are all bases; record starts are invalid entries and every file starts on a
// group boundary behind invalid padding, so no valid window straddles two records or two files, and its genome is
// the genome of the file holding group g.
template <bool SMEM, bool COUNT>
__global__ void __launch_bounds__(kQsThreads)
k_query_scan(const QueryScanParams p) {
    extern __shared__ unsigned long long s_keys[];
    const uint64_t slots = 1ULL << p.slot_bits, smask = slots - 1;
    const unsigned long long* __restrict__ keys = p.keys;
    if (SMEM) {
        for (uint32_t i = threadIdx.x; i < slots; i += kQsThreads) s_keys[i] = p.keys[i];
        __syncthreads();
        keys = s_keys;
    }
    const uint64_t n_groups = (p.scalars[S_STREAM_LEN] + 31) >> 5;
    const uint32_t k = p.k, hs = 64 - p.slot_bits, rc_shift = 2 * (k - 1);
    const unsigned long long kmask = k == 32 ? ~0ULL : ((1ULL << (2 * k)) - 1ULL);
    unsigned long long n_win = 0, n_hit = 0;
    for (uint64_t g = (uint64_t)blockIdx.x * kQsThreads + threadIdx.x; g < n_groups; g += (uint64_t)gridDim.x * kQsThreads) {
        const uint32_t v0 = p.valid[g], vp = g ? p.valid[g - 1] : 0u;
        // valid windows: smear the invalid entries over the k - 1 entries that follow them (the smear of
        // unit_bounds_pair, kept as a copy here so that the build's kernel is compiled exactly as before)
        unsigned long long s = ~((unsigned long long)vp | ((unsigned long long)v0 << 32));
        for (uint32_t c = 1; c < k;) { const uint32_t d = c < k - c ? c : k - c; s |= s << d; c += d; }
        const uint32_t vk = ~(uint32_t)(s >> 32);
        if (!vk) continue;
        n_win += __popc(vk);
        const unsigned long long c0 = p.codes[g], cp = g ? p.codes[g - 1] : 0ULL;
        // the k-mer ending at the last entry of group g - 1 (entries 32 - k .. 31 of cp), then one entry at a time:
        // forward strand first base most significant, reverse complement = complemented entries, oldest least significant
        const unsigned long long v = cp >> (64 - 2 * k);
        unsigned long long fw = rev2_64(v) >> (64 - 2 * k);
        unsigned long long rc = v ^ (0xAAAAAAAAAAAAAAAAULL & kmask);
        uint32_t row = 0xFFFFFFFFu;
#pragma unroll
        for (int e = 0; e < 32; ++e) {
            const unsigned long long b = (c0 >> (2 * e)) & 3ULL;
            fw = ((fw << 2) | b) & kmask;
            rc = (rc >> 2) | ((b ^ 2ULL) << rc_shift);
            if (!((vk >> e) & 1u)) continue;
            const unsigned long long can = fw < rc ? fw : rc;
            uint64_t slot = fmix64(can) >> hs;
            unsigned long long key;
            while ((key = keys[slot]) != kEmptyKey && key != can) slot = (slot + 1) & smask;
            if (key == kEmptyKey) continue;
            ++n_hit;
            if (row == 0xFFFFFFFFu) {                  // the genome row of group g: binary search of the file starts
                const uint64_t pos = g << 5;
                uint32_t lo = 0, hi = p.n_files;
                while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (p.fss[mid] <= pos) lo = mid; else hi = mid; }
                row = p.files[lo].row;
            }
            const uint64_t q = p.idx[slot];
            if (COUNT) {
                atomicAdd(&p.counts[(uint64_t)row * p.qd + q], 1u);
            } else {
                // a repeated k-mer of one genome is the common case: the plain read (racy, but OR is idempotent) saves
                // the atomic when the bit is already set
                const uint32_t gr = p.row0 + row;
                unsigned long long* w = p.plane + (uint64_t)((gr >> 6) - (p.row0 >> 6)) * p.qd + q;
                const unsigned long long bit = 1ULL << (63 - (gr & 63u));
                if (!(*w & bit)) atomicOr(w, bit);
            }
        }
    }
    // one atomic per warp and counter
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n_win += __shfl_down_sync(0xffffffffu, n_win, o);
        n_hit += __shfl_down_sync(0xffffffffu, n_hit, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (n_win) atomicAdd(&p.totals[0], n_win);
        if (n_hit) atomicAdd(&p.totals[1], n_hit);
    }
}

struct QueryGatherParams {
    const unsigned long long* plane;     // presence: [n_words][qd]
    const uint32_t* counts;              // counters: [n_rows][qd]
    const uint32_t* col;                 // [n] plane column of the caller's k-mer i
    uint64_t qd, n;
    uint32_t n_words;                    // word rows the range touches: row0 / 64 .. (row0 + n_rows - 1) / 64
    uint32_t row0, n_rows, min_abundance;
    unsigned long long* out;             // [n_words][n]
};

template <bool COUNT>
__global__ void __launch_bounds__(256)
k_query_gather(const QueryGatherParams p) {
    const uint64_t total = (uint64_t)p.n_words * p.n;
    for (uint64_t t = (uint64_t)blockIdx.x * 256 + threadIdx.x; t < total; t += (uint64_t)gridDim.x * 256) {
        const uint32_t w = (uint32_t)(t / p.n);
        const uint64_t q = p.col[t - (uint64_t)w * p.n];
        if (!COUNT) { p.out[t] = p.plane[(uint64_t)w * p.qd + q]; continue; }
        const uint32_t gw = (p.row0 >> 6) + w;
        const uint32_t r_lo = max(p.row0, gw << 6), r_hi = min(p.row0 + p.n_rows, (gw << 6) + 64u);
        unsigned long long word = 0;
        for (uint32_t r = r_lo; r < r_hi; ++r)
            if (p.counts[(uint64_t)(r - p.row0) * p.qd + q] >= p.min_abundance) word |= 1ULL << (63 - (r & 63u));
        p.out[t] = word;
    }
}

}  // namespace grmkm
