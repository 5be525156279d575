// grmkm_kernels.cuh -- the sm_100a kernels of the k-mer matrix path.
//
//   parse   : k_first_header, k_tile_tickets, k_pack (one pass: tile summaries resolved by decoupled look-back)
//             FASTA/FASTQ text -> dense 2-bit base stream + validity mask   (multidsk's bank reader)
//   units   : grmkm_units.cuh      minimizer-bounded super-k-mers -> content buckets -> dedupe -> k-mer records
//   merge   : k_aggregate_cols     per-bucket shared-memory hash aggregation.  Presence: the bits of all genomes
//             ORed into 64-genome words + singleton filter (dsk2kover); abundance: per-(k-mer, genome) counters
//             and the -abundance-min filter (multidsk); owner-side merge of partial columns (N GPUs)
//   emit    : k_kmer_strings, k_format_tsv                                  (kmer_sequences / Ray TSV)
#pragma once
#include "grmkm_device.cuh"

namespace grmkm {

// ------------------------------------------------------------------------------------------
// parse
// ------------------------------------------------------------------------------------------

// One warp per file: offset of the first header marker ('>' / '@') at a line start, or len.
__global__ void k_first_header(const FileDesc* __restrict__ files, uint32_t n_files, uint64_t* __restrict__ hdr0) {
    const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (f >= n_files) return;
    const FileDesc fd = files[f];
    const uint32_t marker = fd.kind == 0 ? '>' : '@';
    uint64_t found = fd.len;
    for (uint64_t base = 0; base < fd.len; base += 32) {
        const uint64_t pos = base + lane;
        bool hit = false;
        if (pos < fd.len) {
            const uint32_t c = fd.ptr[pos];
            const bool ls = pos == 0 || fd.ptr[pos - 1] == '\n';
            hit = ls && c == marker;
        }
        const uint32_t m = __ballot_sync(0xffffffffu, hit);
        if (m) { found = base + (__ffs(m) - 1); break; }
    }
    if (lane == 0) hdr0[f] = found;
}

struct TileCtx {
    FileDesc fd;
    uint64_t hdr0;
    uint64_t off;   // byte offset of this thread's first chunk in the file (64 contiguous bytes per thread)
    uint32_t f;
    bool first_tile;
};

// the thread's four chunks and the byte before each of them
struct ThreadText {
    Chunk16 ch[kChunksPerThread];
    uint32_t prev[kChunksPerThread];
};
__device__ __forceinline__ ThreadText load_thread_text(const TileCtx& t) {
    ThreadText x;
#pragma unroll
    for (int c = 0; c < kChunksPerThread; ++c) x.ch[c] = load_chunk(t.fd.ptr, t.off + 16 * c, t.fd.len);
    uint32_t p = __shfl_up_sync(0xffffffffu, x.ch[kChunksPerThread - 1].byte(15), 1);
    if ((threadIdx.x & 31) == 0) p = (t.off > 0 && t.off - 1 < t.fd.len) ? t.fd.ptr[t.off - 1] : (uint32_t)'\n';
    x.prev[0] = p;
#pragma unroll
    for (int c = 1; c < kChunksPerThread; ++c) x.prev[c] = x.ch[c - 1].byte(15);
    return x;
}

// Everything a CTA needs to start on ticket t, in one 64-byte record: ticket -> tile (order) -> file -> descriptor,
// first header and stream start used to be four dependent loads at the head of every CTA.
struct TileTicket {
    FileDesc fd;
    uint64_t hdr0;
    uint64_t stream_start;      // where the file's entries start in the packed stream
    uint32_t tile, f;
    uint64_t pad;
};
static_assert(sizeof(TileTicket) == 64, "one ticket = four 16-byte loads");
__global__ void k_tile_tickets(const FileDesc* __restrict__ files, uint32_t n_files, const uint64_t* __restrict__ hdr0,
                               const uint64_t* __restrict__ fss, const uint32_t* __restrict__ order, uint64_t n_tiles,
                               TileTicket* __restrict__ out) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    TileTicket k;
    k.tile = order[t];
    uint32_t lo = 0, hi = n_files - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (files[mid].tile_begin <= k.tile) lo = mid; else hi = mid - 1;
    }
    k.f = lo; k.fd = files[lo]; k.hdr0 = hdr0[lo]; k.stream_start = fss[lo]; k.pad = 0;
    out[t] = k;
}

// ---- single-pass parse: decoupled look-back over the tile summaries --------------------------------------
// The parser is a transducer scan (tile summary = state -> (end state, entries emitted), composition associative).
// Instead of summary kernel + scan kernels + pack kernel (the text read twice), k_pack publishes its tile's
// summary as soon as the block scan has produced it, and one warp walks back over the earlier tiles' published
// summaries until it meets a tile whose incoming (state, position) is already resolved.  Tiles take their index
// from a ticket counter, so every tile a CTA waits for has started and publishes without waiting for anybody.
// Every published word validates itself (bit 63; the arrays are zeroed before the launch), so a reader needs one
// round trip per window of 64 tiles and no fences:
//   a0[t] = 1<<63 | e << 48 | c0 << 24 | c1      summary: end states, entries emitted from state 0 / 1
//   a1[t] = 1<<63 | c2 << 24 | c3                (FASTQ only: states 2 and 3)
//   ps[t] = 1<<63 | state << 61 | position       state and stream position at the tile's first byte
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
constexpr unsigned long long kPubValid = 1ULL << 63;
__device__ __forceinline__ unsigned long long pub_a0(const Sum& s) {
    return kPubValid | ((unsigned long long)(s.e & 0xFFu) << 48) | ((unsigned long long)(s.c0 & 0xFFFFFFu) << 24) | (s.c1 & 0xFFFFFFu);
}
__device__ __forceinline__ unsigned long long pub_a1(const Sum& s) {
    return kPubValid | ((unsigned long long)(s.c2 & 0xFFFFFFu) << 24) | (s.c3 & 0xFFFFFFu);
}
__device__ __forceinline__ Sum pub_sum(unsigned long long a0, unsigned long long a1) {
    Sum r;
    r.e = (uint32_t)(a0 >> 48) & 0xFFu; r.c0 = (uint32_t)(a0 >> 24) & 0xFFFFFFu; r.c1 = (uint32_t)a0 & 0xFFFFFFu;
    r.c2 = (uint32_t)(a1 >> 24) & 0xFFFFFFu; r.c3 = (uint32_t)a1 & 0xFFFFFFu;
    return r;
}
static_assert(kTileBytes < (1 << 24), "a tile's entry counts are published in 24 bits");
__device__ __forceinline__ Sum sum_shfl_down(const Sum& a, int d) {
    Sum r;
    r.e = __shfl_down_sync(0xffffffffu, a.e, d);
    r.c0 = __shfl_down_sync(0xffffffffu, a.c0, d);
    r.c1 = __shfl_down_sync(0xffffffffu, a.c1, d);
    r.c2 = __shfl_down_sync(0xffffffffu, a.c2, d);
    r.c3 = __shfl_down_sync(0xffffffffu, a.c3, d);
    return r;
}
// ordered fold of one Sum per lane (lane 0 first); the result is valid in every lane
template <bool ROT>
__device__ __forceinline__ Sum warp_fold_sum(Sum s) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const Sum o = sum_shfl_down(s, d);
        if (lane + d < 32) s = sum_comb<ROT>(s, o);            // lane i: fold of lanes [i, i + 2d)
    }
    Sum w;
    w.e = __shfl_sync(0xffffffffu, s.e, 0); w.c0 = __shfl_sync(0xffffffffu, s.c0, 0); w.c1 = __shfl_sync(0xffffffffu, s.c1, 0);
    w.c2 = __shfl_sync(0xffffffffu, s.c2, 0); w.c3 = __shfl_sync(0xffffffffu, s.c3, 0);
    return w;
}
// one full warp; state and stream position at the first byte of `tile`.  Every file starts in state 0 at a stream
// position the host fixes in advance (file_stream_start: the file's length rounded up to whole groups bounds its
// entries, the gap reads as invalid entries, and no window spans two files anyway), so the chain of a tile ends at
// its file's first tile: tiles before it count as published (identity) and resolved (state 0, that position).
// Tickets are dealt round-robin over the files (PackParams::order), so the tile a CTA depends on was started one
// whole round earlier and is normally resolved by the time it is asked.
// The counts folded here cover only tiles that are in flight, far below 2^32 entries.
// kLbWindows x 32 tiles are polled per round trip (lane 31 of window 0 = the nearest tile): the resolved front
// trails the newest published tile by (tiles per microsecond) x (poll latency), and a poll that does not reach it
// costs a whole extra round trip.
#ifndef GRMKM_LB_WINDOWS
#define GRMKM_LB_WINDOWS 1          // (2 and 4 windows per poll measured slower once a fold had become cheap: profiles/r02_pack_occupancy_ab.txt)
#endif
constexpr int kLbWindows = GRMKM_LB_WINDOWS;      // FASTA (tile_lookback_fa): many short per-file chains
constexpr int kLbWindowsFq = 2;                   // FASTQ (tile_lookback): one long chain per read set, the resolved front trails further
template <int KIND>
__device__ __noinline__ void tile_lookback(uint64_t tile, uint64_t first, uint64_t pos_first, const unsigned long long* a0,
                                           const unsigned long long* a1, const unsigned long long* ps, uint32_t& st, uint64_t& pos) {
    const int lane = threadIdx.x & 31;
    const unsigned long long ident = kPubValid | (0xE4ULL << 48);      // the identity summary, published
    Sum acc = sum_identity();                      // fold of the tiles between the resolved one and `tile`
    long long hi = (long long)tile - 1;            // nearest tile not folded yet
    while (true) {
        unsigned long long w0[kLbWindowsFq], w1[kLbWindowsFq], wp[kLbWindowsFq];
#pragma unroll
        for (int w = 0; w < kLbWindowsFq; ++w) {
            const long long j = hi - 32 * w - 31 + lane;
            w0[w] = ident; w1[w] = kPubValid; wp[w] = kPubValid | pos_first;
            if (j >= (long long)first) { w0[w] = ld_relaxed_u64(a0 + j); wp[w] = ld_relaxed_u64(ps + j); if (KIND == 1) w1[w] = ld_relaxed_u64(a1 + j); }
        }
        bool done = false;
        int folded = 0;                            // windows of this poll that are folded into acc
#pragma unroll
        for (int w = 0; w < kLbWindowsFq; ++w) {
            const bool rdy_l = (w0[w] & w1[w] & kPubValid) != 0;
            const uint32_t rdy = __ballot_sync(0xffffffffu, rdy_l);
            const uint32_t res = __ballot_sync(0xffffffffu, rdy_l && (wp[w] & kPubValid));
            if (w == 0 && (res >> 31)) {
                // the usual case: the tile right before this one is resolved (no fold; a fold costs ~600 instructions)
                const unsigned long long q0 = __shfl_sync(0xffffffffu, w0[0], 31), q1 = __shfl_sync(0xffffffffu, w1[0], 31);
                const unsigned long long r = __shfl_sync(0xffffffffu, wp[0], 31);
                const Sum a = sum_comb<KIND == 1>(pub_sum(q0, q1), acc);
                const uint32_t st0 = (uint32_t)(r >> 61) & 3u;
                st = sum_end(a, st0);
                pos = (r & ((1ULL << 61) - 1)) + sum_cnt(a, st0);
                return;
            }
            const int top = res ? 31 - __clz(res) : 0;             // nearest resolved tile of the window, if any
            if ((rdy >> top) != (0xFFFFFFFFu >> top)) break;       // a tile this side of it has not published yet: poll again
            acc = sum_comb<KIND == 1>(warp_fold_sum<KIND == 1>(lane < top ? sum_identity() : pub_sum(w0[w], w1[w])), acc);
            folded = w + 1;
            if (res) {
                const unsigned long long r = __shfl_sync(0xffffffffu, wp[w], top);
                const uint32_t st0 = (uint32_t)(r >> 61) & 3u;
                st = sum_end(acc, st0);
                pos = (r & ((1ULL << 61) - 1)) + sum_cnt(acc, st0);
                done = true;
                break;
            }
        }
        if (done) return;
        hi -= 32 * folded;
    }
}

// FASTA: the same walk with the summaries in their compact form (grmkm_device.cuh, fa_combine) widened to 64 bits --
// bits 0-29 entries after the first line start, 30-59 sequence bytes before it, 60-61 type of the last line start.  A
// fold of 32 summaries is then ~70 instructions instead of ~600 with the general four-state transducer, so a tile
// whose predecessor is not resolved yet folds from an older resolved tile instead of waiting a round trip per hop.
__device__ __forceinline__ unsigned long long fa64_from_pub(unsigned long long a0) {
    const uint32_t e = (uint32_t)(a0 >> 48) & 0xFFu, c0 = (uint32_t)(a0 >> 24) & 0xFFFFFFu, c1 = (uint32_t)a0 & 0xFFFFFFu;
    const unsigned long long t = e == 0xE4u ? 0ULL : (unsigned long long)((e & 3u) + 1u);
    return (unsigned long long)c0 | ((unsigned long long)(c1 - c0) << 30) | (t << 60);
}
__device__ __forceinline__ unsigned long long fa64_combine(unsigned long long A, unsigned long long B) {      // A first, then B
    constexpr unsigned long long M30 = (1ULL << 30) - 1;
    const uint32_t ta = (uint32_t)(A >> 60), tb = (uint32_t)(B >> 60);
    const unsigned long long hb = (B >> 30) & M30;
    unsigned long long r = (A & ((1ULL << 60) - 1)) + (B & M30);
    r += ta == 0 ? hb << 30 : 0ULL;
    r += ta == 2 ? hb : 0ULL;
    return r | ((unsigned long long)(tb ? tb : ta) << 60);
}
__device__ __noinline__ void tile_lookback_fa(uint64_t tile, uint64_t first, uint64_t pos_first, const unsigned long long* a0,
                                              const unsigned long long* ps, uint32_t& st, uint64_t& pos) {
    constexpr unsigned long long M30 = (1ULL << 30) - 1;
    const int lane = threadIdx.x & 31;
    const unsigned long long ident = kPubValid | (0xE4ULL << 48);
    unsigned long long acc = 0;                    // fold of the tiles between the resolved one and `tile` (identity: nothing seen)
    long long hi = (long long)tile - 1;
    auto finish = [&](unsigned long long r, unsigned long long a) {
        const uint32_t st0 = (uint32_t)(r >> 61) & 3u, t = (uint32_t)(a >> 60);
        st = t ? t - 1u : st0;
        pos = (r & ((1ULL << 61) - 1)) + (a & M30) + (st0 == ST_SEQ ? ((a >> 30) & M30) : 0ULL);
    };
    while (true) {
        unsigned long long w0[kLbWindows], wp[kLbWindows];
#pragma unroll
        for (int w = 0; w < kLbWindows; ++w) {
            const long long j = hi - 32 * w - 31 + lane;
            w0[w] = ident; wp[w] = kPubValid | pos_first;
            if (j >= (long long)first) { w0[w] = ld_relaxed_u64(a0 + j); wp[w] = ld_relaxed_u64(ps + j); }
        }
        int folded = 0;
#pragma unroll
        for (int w = 0; w < kLbWindows; ++w) {
            const bool rdy_l = (w0[w] & kPubValid) != 0;
            const uint32_t rdy = __ballot_sync(0xffffffffu, rdy_l);
            const uint32_t res = __ballot_sync(0xffffffffu, rdy_l && (wp[w] & kPubValid));
            if (w == 0 && (res >> 31)) {                           // the usual case: the tile right before this one is resolved
                finish(__shfl_sync(0xffffffffu, wp[0], 31), fa64_combine(fa64_from_pub(__shfl_sync(0xffffffffu, w0[0], 31)), acc));
                return;
            }
            const int top = res ? 31 - __clz(res) : 0;             // nearest resolved tile of the window, if any
            if ((rdy >> top) != (0xFFFFFFFFu >> top)) break;       // a tile this side of it has not published yet: poll again
            // ordered fold of lanes top .. 31 (lane 31 = the nearest tile); lanes below top count as the identity
            unsigned long long v = lane < top ? 0ULL : fa64_from_pub(w0[w]);
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned long long o = __shfl_down_sync(0xffffffffu, v, d);
                if (lane + d < 32) v = fa64_combine(v, o);
            }
            acc = fa64_combine(__shfl_sync(0xffffffffu, v, 0), acc);
            folded = w + 1;
            if (res) {
                finish(__shfl_sync(0xffffffffu, wp[w], top), acc);
                return;
            }
        }
        hi -= 32 * folded;
    }
}

// text tile -> packed stream: codes64[g] holds entries 32g..32g+31 (entry j at bits 2j), valid32[g] bit j.
// Every thread turns its 64 bytes into at most 64 entries (register accumulator), the block scan of the
// thread summaries gives each thread its entry offset inside the tile, the look-back gives the tile its state and
// position, and the tile is assembled in shared memory.
struct PackParams {
    const FileDesc* files;
    const uint64_t* hdr0;
    uint64_t n_tiles;
    uint32_t n_files;
    const TileTicket* tickets;          // [n_tiles] ticket -> tile and its file, tickets dealt round-robin over the files
    uint64_t stream_len;                // padded stream length of the batch (-> scalars[S_STREAM_LEN])
    uint32_t* ticket;                   // zeroed before the launch
    unsigned long long* pub_a0;         // [n_tiles] x 3, zeroed before the launch (see tile_lookback)
    unsigned long long* pub_a1;
    unsigned long long* pub_ps;
    unsigned long long* codes;
    uint32_t* valid;
    uint64_t* scalars;
};

template <int KIND>
#ifndef GRMKM_PACK_CTAS
#define GRMKM_PACK_CTAS (1024 / kParseThreads)      // resident CTAs per SM the register budget is cut for (A/B: profiles/r02_pack_occupancy_ab.txt)
#endif
__global__ void __launch_bounds__(kParseThreads, GRMKM_PACK_CTAS)
k_pack(const PackParams p) {
    constexpr int kGroups = kTileBytes / 32 + 2;
    __shared__ Sum s_w[2 * (kParseThreads / 32) + 1];
    // the tile's groups, assembled with shared-memory ORs: codes (two words per group) and validity bits in ONE 16-byte
    // aligned block, so that it is cleared with two 128-bit stores per thread
    constexpr int kCodeWords = kGroups * 2 + 4, kValidWords = kGroups + 2;
    constexpr int kCvVec = (kCodeWords + kValidWords + 3) / 4;
    static_assert(kCodeWords % 4 == 0, "the validity words start on a 16-byte boundary");
    __shared__ __align__(16) uint32_t s_cv[kCvVec * 4];
    uint32_t* const s_codes = s_cv;
    uint32_t* const s_valid = s_cv + kCodeWords;
    __shared__ uint32_t s_nrec, s_st;
    __shared__ uint64_t s_pos;
    __shared__ uint4 s_tk[4];                                           // this CTA's TileTicket
    // ---- one tile per CTA, tickets from the counter
    if (threadIdx.x == 0) {
        const uint32_t ticket = atomicAdd(p.ticket, 1u);
        s_nrec = 0;
        if (ticket == 0) p.scalars[S_STREAM_LEN] = p.stream_len;
        if (ticket < p.n_tiles) {
            const uint4* src = reinterpret_cast<const uint4*>(p.tickets + ticket);
            const uint4 a = src[0], b = src[1], c = src[2], d = src[3];
            s_tk[0] = a; s_tk[1] = b; s_tk[2] = c; s_tk[3] = d;
        } else {
            s_tk[3] = make_uint4(0xFFFFFFFFu, 0u, 0u, 0u);                 // no tile left
        }
    }
    for (int i = threadIdx.x; i < kCvVec; i += kParseThreads) reinterpret_cast<uint4*>(s_cv)[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const TileTicket& tk = *reinterpret_cast<const TileTicket*>(s_tk);
    if (tk.tile == 0xFFFFFFFFu) return;
    TileCtx t;
    t.f = tk.f; t.fd = tk.fd; t.hdr0 = tk.hdr0;
    t.first_tile = (tk.tile == t.fd.tile_begin);
    t.off = (tk.tile - t.fd.tile_begin) * (uint64_t)kTileBytes + (uint64_t)threadIdx.x * (16 * kChunksPerThread);
    const ThreadText x = load_thread_text(t);
    // ---- everything after the thread's 64 bytes are in registers
    const uint64_t tile = tk.tile;
    unsigned long long* __restrict__ codes = p.codes;
    uint32_t* __restrict__ valid = p.valid;
    const uint64_t file_stream_start = tk.stream_start;
    // publish the tile's summary, resolve its incoming state and position (warp 0), publish those
    auto publish = [&](const Sum& total) {
        if (threadIdx.x == 0) {
            if (KIND == 1) st_relaxed_u64(p.pub_a1 + tile, pub_a1(total));
            st_relaxed_u64(p.pub_a0 + tile, pub_a0(total));
        }
    };
    auto resolve = [&](uint32_t& st_in, uint64_t& tpos) {
        if (threadIdx.x < 32) {
            uint32_t st; uint64_t pos;
            if (KIND == 0) tile_lookback_fa(tile, t.fd.tile_begin, file_stream_start, p.pub_a0, p.pub_ps, st, pos);
            else tile_lookback<KIND>(tile, t.fd.tile_begin, file_stream_start, p.pub_a0, p.pub_a1, p.pub_ps, st, pos);
            if (threadIdx.x == 0) {
                st_relaxed_u64(p.pub_ps + tile, kPubValid | ((unsigned long long)st << 61) | pos);
                s_st = st; s_pos = pos;
            }
        }
        __syncthreads();
        st_in = s_st; tpos = s_pos;
    };
    uint32_t st_in; uint64_t tpos;
    Acc64 acc; acc.init();
    uint32_t nrec = 0, local, e_total;
    if (KIND == 0) {
        FaParts part[kChunksPerThread];
        uint32_t mine = 0;
#pragma unroll
        for (int c = 0; c < kChunksPerThread; ++c) {
            const FaLines ln = fa_lines(x.ch[c], t.off + 16 * c, t.fd.len, t.hdr0);
            part[c] = fa_chunk_parts(x.ch[c], ln, x.prev[c], t.off + 16 * c, t.fd.len, t.hdr0);
            mine = fa_combine(mine, part[c].sum());
        }
        uint32_t ex, tot;
        block_scan_fa(mine, ex, tot, reinterpret_cast<uint32_t*>(s_w));
        publish(fa_to_sum(tot));
        // The entries are accumulated while the look-back is still in flight, as if the tile started inside a sequence
        // line; the few threads in front of the tile's first line start redo it when it started inside a header.
        const uint32_t ex_t = ex >> kFaT;
        auto build = [&](bool in_seq) {                              // in_seq: line type at this thread's first byte
            acc.init(); nrec = 0;
#pragma unroll
            for (int c = 0; c < kChunksPerThread; ++c) {
                // head (only inside a sequence line) and rest of the chunk as ONE run of at most 16 entries
                const uint32_t hn = in_seq ? part[c].hn() : 0u;
                const uint32_t cc = (in_seq ? part[c].hc : 0u) | (hn < 16u ? part[c].rc << (2 * hn) : 0u);      // hn = 16: no rest
                const uint32_t vv = (in_seq ? part[c].hv_rv & 0xFFFFu : 0u) | ((part[c].hv_rv >> 16) << hn);
                acc.append(cc, vv, hn + part[c].rn());
                nrec += part[c].nrec();
                if (part[c].t()) in_seq = (part[c].t() == 2);
            }
        };
        build(ex_t ? (ex_t == 2) : true);
        resolve(st_in, tpos);
        const bool tile_seq = (st_in == ST_SEQ);
        if (!tile_seq && ex_t == 0) build(false);
        local = (ex & kFaMask) + (tile_seq ? ((ex >> kFaH) & kFaMask) : 0u);
        e_total = (tot & kFaMask) + (tile_seq ? ((tot >> kFaH) & kFaMask) : 0u);
    } else {
        // A live chunk whose only control characters are newlines is classified without a byte loop (fq_lines /
        // fq_summary): nine chunks of ten of 150-base reads hold no newline at all, the rest one or two.  Byte loops
        // are left for CR-LF text, tabs and the first / last bytes of a file.
        Sum sums[kChunksPerThread];
        Sum mine = sum_identity(), excl, total;
        uint32_t fastm = 0, nlm[kChunksPerThread];
#pragma unroll
        for (int c = 0; c < kChunksPerThread; ++c) {
            const uint64_t pos0 = t.off + 16 * c;
            uint32_t ctrl;
            fq_control(x.ch[c], ctrl, nlm[c]);
            if (ctrl == nlm[c] && pos0 >= t.hdr0 && pos0 + 16 <= t.fd.len) {
                fastm |= 1u << c;
                const bool first = pos0 == t.hdr0 || x.prev[c] == '\n';
                if (nlm[c] == 0) { sums[c].e = 0xE4u; sums[c].c0 = first ? 1u : 0u; sums[c].c1 = 16u; sums[c].c2 = sums[c].c3 = 0u; }
                else sums[c] = fq_summary(fq_lines(nlm[c], first));
            } else {
                sums[c] = chunk_summary<1>(x.ch[c], x.prev[c], pos0, t.fd.len, t.hdr0);
            }
            mine = sum_combine_rot(mine, sums[c]);
        }
        block_scan_sum<true>(mine, excl, total, s_w);
        publish(total);
        resolve(st_in, tpos);
        uint32_t st = sum_end(excl, st_in);
        local = sum_cnt(excl, st_in);
        e_total = sum_cnt(total, st_in);
#pragma unroll
        for (int c = 0; c < kChunksPerThread; ++c) {
            if ((fastm >> c) & 1u) {
                const bool first = (t.off + 16 * c) == t.hdr0 || x.prev[c] == '\n';
                if (nlm[c] == 0) {
                    if (st == 1) {
                        uint32_t vb, cb;
                        fa_bases(x.ch[c], vb, cb);
                        acc.append(cb, vb, 16u);
                    } else if (st == 0 && first) { acc.append(0u, 0u, 1u); nrec++; }
                    continue;
                }
                const FqChunk f = fq_lines(nlm[c], first);
                const uint32_t nn = ~f.nl & 0xFFFFu;
                const uint32_t seq = fq_line_mask(f, (1u - st) & 3u) & nn;          // bytes of the sequence line
                const uint32_t hdr = fq_line_mask(f, (4u - st) & 3u) & nn & f.ls;   // first bytes of header lines
                uint32_t vb = 0, cb = 0;
                if (seq) { fa_bases(x.ch[c], vb, cb); vb &= seq; }
                nrec += (uint32_t)__popc(hdr);
                for (uint32_t em = seq | hdr; em;) {               // runs of emitting bytes (one, seldom two)
                    const uint32_t s0 = (uint32_t)__ffs(em) - 1u;
                    const uint32_t run = (uint32_t)__ffs(~(em >> s0)) - 1u;
                    const uint32_t lo = (1u << run) - 1u;
                    acc.append((cb >> (2u * s0)) & (run >= 16u ? 0xFFFFFFFFu : ((1u << (2u * run)) - 1u)), (vb >> s0) & lo, run);
                    em &= ~(lo << s0);
                }
                st = (st + (uint32_t)__popc(f.nl)) & 3u;
                continue;
            }
            uint32_t cbits = 0, vbits = 0, n = 0, prev = x.prev[c];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const uint64_t pos = t.off + 16 * c + i;
                const uint32_t ch = x.ch[c].byte(i);
                if (pos < t.fd.len && pos >= t.hdr0) {
                    const bool ls = (pos == t.hdr0) || (prev == '\n');
                    if (ch == '\n') st = (st + 1) & 3;
                    else if (st == 0) { if (ls) { n++; nrec++; } }
                    else if (st == 1 && ch != '\r') {
                        if (is_acgt(ch)) { cbits |= ((ch >> 1) & 3u) << (2 * n); vbits |= 1u << n; }
                        n++;
                    }
                }
                prev = ch;
            }
            acc.append(cbits, vbits, n);
        }
    }
    if (acc.n) {
        const uint32_t rel = (uint32_t)(tpos & 31) + local;         // entry offset from the tile's first group
        const uint32_t cb = rel * 2, cw = cb >> 5, cs = cb & 31;
        const uint32_t c0 = (uint32_t)acc.clo, c1 = (uint32_t)(acc.clo >> 32), c2 = (uint32_t)acc.chi, c3 = (uint32_t)(acc.chi >> 32);
        const uint32_t w0 = c0 << cs, w1 = __funnelshift_l(c0, c1, cs), w2 = __funnelshift_l(c1, c2, cs),
                       w3 = __funnelshift_l(c2, c3, cs), w4 = cs ? (c3 >> (32 - cs)) : 0u;
        if (w0) atomicOr(&s_codes[cw], w0);
        if (w1) atomicOr(&s_codes[cw + 1], w1);
        if (w2) atomicOr(&s_codes[cw + 2], w2);
        if (w3) atomicOr(&s_codes[cw + 3], w3);
        if (w4) atomicOr(&s_codes[cw + 4], w4);
        const uint32_t vw = rel >> 5, vs = rel & 31;
        const uint32_t v0 = (uint32_t)acc.v, v1 = (uint32_t)(acc.v >> 32);
        const uint32_t u0 = v0 << vs, u1 = __funnelshift_l(v0, v1, vs), u2 = vs ? (v1 >> (32 - vs)) : 0u;
        if (u0) atomicOr(&s_valid[vw], u0);
        if (u1) atomicOr(&s_valid[vw + 1], u1);
        if (u2) atomicOr(&s_valid[vw + 2], u2);
    }
    if (nrec) atomicAdd(&s_nrec, nrec);
    __syncthreads();
    if (e_total) {
        // groups [lo, hi) belong to this tile alone: plain stores; the first group (when the tile starts inside it) and
        // the last one (when it ends inside it) are shared with the neighbouring tiles and ORed into the zeroed stream
        const uint64_t g0 = tpos >> 5;
        const uint32_t first_off = (uint32_t)(tpos & 31), end_off = first_off + e_total;
        const uint32_t lo = first_off ? 1u : 0u, hi = end_off >> 5;
        const unsigned long long* __restrict__ sc64 = reinterpret_cast<const unsigned long long*>(s_codes);
        for (uint32_t gi = lo + threadIdx.x; gi < hi; gi += kParseThreads) {
            codes[g0 + gi] = sc64[gi];
            valid[g0 + gi] = s_valid[gi];
        }
        uint32_t pg = 0xFFFFFFFFu;
        if (threadIdx.x == 0 && first_off) pg = 0;
        if (threadIdx.x == 32 && (end_off & 31u) && (hi > 0 || !first_off)) pg = hi;
        if (pg != 0xFFFFFFFFu) {
            const unsigned long long cw = sc64[pg];
            const uint32_t vw = s_valid[pg];
            if (cw) atomicOr(&codes[g0 + pg], cw);
            if (vw) atomicOr(&valid[g0 + pg], vw);
        }
    }
    if (threadIdx.x == 0) {
        if (s_nrec) atomicAdd((unsigned long long*)&p.scalars[S_N_RECORDS], (unsigned long long)s_nrec);
        if (e_total) atomicAdd((unsigned long long*)&p.scalars[S_STREAM_TOTAL], (unsigned long long)e_total);
    }
}

// ---- tile sort of hashed k-mers (k_units_expand): one tile = kStThreads x kStPerThread k-mers per CTA iteration;
// tile histogram with shared-memory atomics, ONE global reservation per (tile, bucket), counting sort in shared
// memory, bucket runs on the way out.  Bucket regions are exact (cursors = prefix sums of a count pass) or
// over-provisioned (region b = [b * cap, (b + 1) * cap)); an overflowing bucket raises a flag and its records go
// to a dump area, the host then re-runs with exact offsets.
constexpr int kStThreads = 512;                        // (1024 threads, two per unit with 16 k-mers each, were measured: expand
                                                       // 0.218 -> 0.283 ms: the unit decode runs twice and the barriers get wider)
constexpr int kStPerThread = 32;                       // up to 32 k-mers per thread
constexpr int kStTile = kStThreads * kStPerThread;     // 16384 positions = 512 groups
constexpr int kStMaxBuckets = 4096;
constexpr int kStMaxBins = kStMaxBuckets / kStThreads; // bins per thread in phase 2

__host__ __device__ inline size_t staged_smem_bytes(uint32_t B) {
    return (size_t)B * (8 + 4 + 4) + (size_t)kStTile * (8 + 2);
}

__device__ __forceinline__ uint32_t rev2_32(uint32_t x) {
    x = __brev(x);
    return ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
}

// exclusive scan of one u32 per thread over an NT-thread block; s_warp must hold 33 words
template <int NT>
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t* s_warp, uint32_t& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < NT / 32 ? s_warp[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, wi, d);
            if (lane >= d) wi += o;
        }
        s_warp[lane] = wi - w;          // exclusive warp offsets
        if (lane == 31) s_warp[32] = wi;
    }
    __syncthreads();
    total = s_warp[32];
    const uint32_t r = s_warp[warp] + inc - v;
    __syncthreads();
    return r;
}

// sum of one u64 per thread over a block of up to 1024 threads (valid in thread 0); a 64-bit atomicAdd on shared
// memory is a compare-and-swap loop, 1024 of them on one word took 40 us
__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v) {
    __shared__ unsigned long long s_part[32];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    if ((threadIdx.x & 31u) == 0) s_part[threadIdx.x >> 5] = v;
    __syncthreads();
    unsigned long long t = 0;
    if (threadIdx.x < 32) {
        t = threadIdx.x < (blockDim.x + 31) / 32 ? s_part[threadIdx.x] : 0ULL;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) t += __shfl_down_sync(0xffffffffu, t, d);
    }
    return t;
}

// After the scatter: end[b] = cursor[b], clamped to the region when regions are over-provisioned (an
// overflowing bucket is re-done by the exact path, but nothing may read past its region meanwhile);
// scalars[which] = number of records = n_windows.  One block.
__global__ void __launch_bounds__(1024)
k_finish_regions(const unsigned long long* __restrict__ begin, unsigned long long* __restrict__ end, uint32_t B,
                 unsigned long long cap, unsigned long long* __restrict__ scalars, int which) {
    unsigned long long v = 0;
    for (uint32_t b = threadIdx.x; b < B; b += blockDim.x) {
        unsigned long long e = end[b];
        if (cap && e > (unsigned long long)(b + 1) * cap) { e = (unsigned long long)(b + 1) * cap; end[b] = e; }
        v += e - begin[b];
    }
    const unsigned long long sum = block_sum_u64(v);
    if (threadIdx.x == 0) scalars[which] = sum;
}

// region starts for the over-provisioned layout: begin[b] = cursors[b] = b * cap
__global__ void k_init_regions(unsigned long long* __restrict__ begin, unsigned long long* __restrict__ cursors,
                               uint32_t B, unsigned long long cap) {
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) { begin[b] = (unsigned long long)b * cap; cursors[b] = (unsigned long long)b * cap; }
    if (b == B) begin[b] = (unsigned long long)B * cap;
}

// exclusive scan of the bucket histogram -> offsets[B+1]; cursors[b] = offsets[b]
__global__ void __launch_bounds__(1024)
k_bucket_offsets(unsigned long long* __restrict__ hist_cursor, unsigned long long* __restrict__ offsets, uint32_t B,
                 uint64_t* __restrict__ scalars, int total_scalar, uint32_t stride) {
    __shared__ unsigned long long s_part[1024];
    const uint32_t per = (B + 1023) / 1024;
    const uint32_t b0 = threadIdx.x * per;
    unsigned long long sum = 0;
    for (uint32_t i = 0; i < per; ++i) if (b0 + i < B) sum += hist_cursor[(size_t)(b0 + i) * stride];
    s_part[threadIdx.x] = sum;
    __syncthreads();
    // simple Hillis-Steele inclusive scan
    for (int d = 1; d < 1024; d <<= 1) {
        unsigned long long v = threadIdx.x >= d ? s_part[threadIdx.x - d] : 0;
        __syncthreads();
        s_part[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned long long run = s_part[threadIdx.x] - sum;
    for (uint32_t i = 0; i < per; ++i) {
        if (b0 + i < B) {
            const unsigned long long c = hist_cursor[(size_t)(b0 + i) * stride];
            offsets[b0 + i] = run;
            hist_cursor[(size_t)(b0 + i) * stride] = run;
            run += c;
        }
    }
    if (threadIdx.x == 1023) { offsets[B] = s_part[1023]; scalars[total_scalar] = s_part[1023]; }
}

// ---- column aggregation: MODE 4 = final columns, 5 = partial columns (N GPUs), 3 = owner-side merge of partial
// columns, 6 = abundance round (per-genome counters -> solid presence records), 7 = pooled count table ----
// One CTA per hash bucket.  The bucket's records stream through a shared-memory table
//   keys[slots + tail] (u64), w32[2W][slots + tail] (presence half-words), kept[slots + tail] (u8)
// with eight coalesced loads in flight per thread.  Genome row g lives in half-word plane (g >> 5) ^ 1 at bit
// 31 - (g & 31), so that word w = w32[2w+1] : w32[2w] has row g at bit 63 - (g & 63) (kover/utils.py:144-154).
//
// The home slot is MONOTONE in the key (its top bits scaled to the table; the multiplicative hash already
// spreads them uniformly) and probing never wraps (tail slots), so clusters hold disjoint ascending key ranges:
// the table is almost sorted, and a key's exact rank is (kept slots before it) corrected by the inversions
// inside its own cluster.  Columns therefore leave the kernel in ascending hash order per bucket with no
// sort pass.  A bucket that does not fit is split into key sub-ranges (processed in ascending order): one
// counting sweep to size the bucket's output, one emitting sweep.
constexpr int kAggBatch = 8;

struct AggTable {
    unsigned long long* keys;
    uint32_t* w32;
    uint8_t* kept;         // [total rounded up to 4] bit 7: the slot's column is kept; bits 0-6: inversions found by LATER slots
    uint8_t* dec;          // [total] inversions the slot found itself (larger kept keys between its home and itself)
    uint32_t slots;        // home slots
    uint32_t total;        // slots + tail
};

__device__ __forceinline__ uint32_t home_slot(unsigned long long key, uint32_t shift, uint32_t slots) {
    // top 32 bits of the key below the bits that are fixed inside the current (sub-)range; shift = 64 - key_bits + depth
    return __umulhi((uint32_t)((key << shift) >> 32), slots);
}

struct AggParams2 {
    const unsigned long long* records;   // MODE 4-7: wide records [(hash << row_bits) | group, words]; MODE 3: unused (parts / bounds)
    const unsigned long long* begin;     // [B]
    const unsigned long long* end;       // [B]
    uint32_t bucket_bits, row_bits, n_words, slots, keep_singletons;
    uint32_t sub_bits;                   // every bucket is aggregated as 2^sub_bits key sub-ranges (virtual buckets), one CTA pass each
    uint32_t wide_words, wide_stride;    // MODE 4/5: presence words per wide record, u64 per record
    uint32_t table_u32;                  // u32 cells per table slot: 2 x n_words presence half-words; MODE 3: one entry reference per source (even)
    unsigned long long* out_keys;        // [cap]   bucket chunks, at bucket_base[b]
    unsigned long long* out_words;       // [n_words][cap]
    unsigned long long cap;
    unsigned long long* scalars;
    unsigned long long* bucket_base;     // [B] where the bucket's chunk starts in out_*
    unsigned long long* bucket_count;    // [B] columns the bucket emitted
    uint32_t b_begin, b_end;             // bucket_base / bucket_count are indexed by (virtual bucket) - (b_begin << sub_bits)
    // ordered emission (final build in hash order): the virtual buckets are dealt by ticket, every bucket publishes its
    // column count and learns its offset by look-back over its predecessors, so the columns land at their final place:
    // out_keys is the result's k-mer array and out_words the result matrix, whose row pitch is cap (the number of
    // columns is only known at the end; every reader of the result takes the pitch)
    uint32_t ordered;
    unsigned long long* pub;             // [virtual buckets] bit 63: inclusive prefix, bit 62: own count; zeroed before the launch
    unsigned int* ticket;                // zeroed before the launch
    // MODE 3: partial columns [hash, words...] of n_src sources, each list ascending by hash; the entries of
    // bucket b in source s are bounds[s * (b_end - b_begin + 1) + (b - b_begin)] .. [.. + 1]
    const unsigned long long* parts;
    const unsigned long long* bounds;
    uint32_t n_src;
    // MODE 6 / 7 (abundance): the table planes are u32 COUNTERS, one per genome row of the round (records
    // [(hash << row_bits) | local row, count]); a row is solid when its counter reaches min_abundance (multidsk
    // -abundance-min, kmer_count.py:48).  MODE 6 emits the round's solid presence as wide records of ONE word
    // [(hash << out_wbits) | out_word, bits] for the final presence aggregate; MODE 7 (pooled counts, src/app.py:1372)
    // emits (k-mer, count of local row 0).
    uint32_t min_abundance, round_rows, round_row0, out_wbits, out_word;
    ulonglong2* out_wide;
    uint32_t partial_out;                // MODE 3: emit partial columns again (hash keys; the caller sets keep_singletons)
    unsigned long long src_off[16];      // first u64 word of the source in parts
    uint32_t src_words[16];
    uint32_t src_woff[16];
};

// Probe loops split warps: a lane that finds its slot at the first probe does not wait for its neighbours by itself,
// and everything after the loop would then run once per fragment (4.2 fragments per warp were measured,
// profiles/r01_v3).  So every lane of the warp runs every iteration of the record loops (inactive ones predicated
// off) and the warp is re-converged with __syncwarp() right after each probe loop.
__device__ __forceinline__ bool agg_insert(unsigned long long* keys, uint32_t& slot, unsigned long long key, bool active) {
    bool ok = active;
    if (active) {
        int probe = 0;
        while (true) {
            unsigned long long k0 = *(volatile unsigned long long*)&keys[slot];
            if (k0 == key) break;
            if (k0 == kEmptyKey) {
                k0 = atomicCAS(&keys[slot], kEmptyKey, key);
                if (k0 == kEmptyKey || k0 == key) break;
            }
            ++slot;
            if (++probe >= kMaxProbe) { ok = false; break; }
        }
    }
    __syncwarp();
    return ok;
}

// MODE 4 / 5: wide records [(hash << row_bits) | genome group, wide_words presence words (, padding)] of
// wide_stride u64 each (the unit path, grmkm_units.cuh); the words of group g are matrix words g * wide_words ..
template <bool FILTER, bool COUNTS>
__device__ __forceinline__ void agg_stream_wide(const AggParams2& p, const AggTable& t, const unsigned long long* __restrict__ recs,
                                                uint32_t n, uint32_t key_bits, uint32_t depth, unsigned long long ridx,
                                                volatile uint32_t* overflow) {
    const uint32_t wbits = p.row_bits;
    const uint32_t wmask = (1u << wbits) - 1u;
    const uint32_t shift = 64 - key_bits + depth;
    const uint32_t slots = t.slots, total = t.total;
    const uint32_t WB = p.wide_words, stride2 = p.wide_stride / 2;          // record = stride2 x 16 bytes
    unsigned long long* const keys = t.keys;
    uint32_t* const w32 = t.w32;
    const ulonglong2* const rec2 = reinterpret_cast<const ulonglong2*>(recs);
    constexpr int kWideBatch = 4;
    for (uint32_t base0 = 0; base0 < n; base0 += kAggThreads * kWideBatch) {
        const uint32_t base = base0 + threadIdx.x;
        ulonglong2 r[kWideBatch], r2[kWideBatch];                  // [key, word 0], [word 1, word 2]
#pragma unroll
        for (int j = 0; j < kWideBatch; ++j) {
            const uint32_t idx = base + j * kAggThreads;
            r[j] = idx < n ? __ldcs(rec2 + (size_t)idx * stride2) : make_ulonglong2(0ULL, 0ULL);
            r2[j] = (idx < n && WB > 1) ? __ldcs(rec2 + (size_t)idx * stride2 + 1) : make_ulonglong2(0ULL, 0ULL);
        }
        if (__any_sync(0xffffffffu, *overflow != 0)) break;
#pragma unroll
        for (int j = 0; j < kWideBatch; ++j) {
            const uint32_t idx = base + j * kAggThreads;
            const unsigned long long key = r[j].x >> wbits;
            bool act = idx < n;
            if (FILTER) act = act && ((key << (64 - key_bits)) >> (64 - depth)) == ridx;
            uint32_t slot = home_slot(key, shift, slots);
            const bool ok = agg_insert(keys, slot, key, act);
            if (act) {
                if (ok && COUNTS) {
                    // abundance: the record's word is the number of occurrences it stands for
                    atomicAdd(&w32[((uint32_t)r[j].x & wmask) * total + slot], (uint32_t)r[j].y);
                } else if (ok) {
                    const uint32_t w0 = ((uint32_t)r[j].x & wmask) * WB;
                    {
                        const uint32_t vlo = (uint32_t)r[j].y, vhi = (uint32_t)(r[j].y >> 32);
                        if (vlo) atomicOr(&w32[(2 * w0) * total + slot], vlo);
                        if (vhi) atomicOr(&w32[(2 * w0 + 1) * total + slot], vhi);
                    }
                    for (uint32_t w = 1; w < WB; ++w) {
                        const unsigned long long v = w == 1 ? r2[j].x : w == 2 ? r2[j].y : __ldcs(recs + (size_t)idx * p.wide_stride + 1 + w);
                        const uint32_t vlo = (uint32_t)v, vhi = (uint32_t)(v >> 32);
                        if (vlo) atomicOr(&w32[(2 * (w0 + w)) * total + slot], vlo);
                        if (vhi) atomicOr(&w32[(2 * (w0 + w) + 1) * total + slot], vhi);
                    }
                } else *overflow = 1;
            }
        }
    }
}

// MODE 3: the bucket's entries are one contiguous range per source (the lists arrive sorted by hash)
template <bool FILTER>
__device__ __forceinline__ void agg_stream_parts(const AggParams2& p, const AggTable& t, uint32_t b, uint32_t key_bits,
                                                 uint32_t depth, unsigned long long ridx, volatile uint32_t* overflow) {
    const uint32_t shift = 64 - key_bits + depth;
    const unsigned long long key_mask = (1ULL << key_bits) - 1;
    const uint32_t nb1 = p.b_end - p.b_begin + 1;
    for (uint32_t s = 0; s < p.n_src; ++s) {
        const unsigned long long lo = p.bounds[(size_t)s * nb1 + (b - p.b_begin)], hi = p.bounds[(size_t)s * nb1 + (b - p.b_begin) + 1];
        const uint32_t width = 1 + p.src_words[s];
        const unsigned long long* src = p.parts + p.src_off[s];
        for (unsigned long long i0 = lo; i0 < hi; i0 += kAggThreads) {
            if (__any_sync(0xffffffffu, *overflow != 0)) break;
            const unsigned long long i = i0 + threadIdx.x;
            bool act = i < hi;
            const unsigned long long* ent = src + (act ? i : lo) * width;
            const unsigned long long key = ent[0] & key_mask;
            if (FILTER) act = act && (key >> (key_bits - depth)) == ridx;
            uint32_t slot = home_slot(key, shift, t.slots);
            const bool ok = agg_insert(t.keys, slot, key, act);
            if (act && !ok) *overflow = 1;
            // the slot keeps a REFERENCE to the source's entry (a source lists a key once), not its words: with 16 word-rows a
            // slot of words is 137 bytes, a slot of 8 references 41, so the table holds 3.3 x the keys and the owner needs
            // that many fewer bucket passes (N = 8: merge 1.9 ms with words in the table)
            if (act && ok) t.w32[s * t.total + slot] = (uint32_t)i + 1u;
        }
    }
}

// bounds[s][j] = first entry of source s whose hash is >= (b_begin + j) << key_bits  (j = 0 .. nb; j with
// b_begin + j == 2^bucket_bits means "the end")
__global__ void k_merge_bounds(const unsigned long long* __restrict__ parts, uint32_t n_src, uint32_t nb1, uint32_t b_begin,
                               uint32_t bucket_bits, const unsigned long long* __restrict__ src_off,
                               const unsigned long long* __restrict__ src_count, const uint32_t* __restrict__ src_width,
                               unsigned long long* __restrict__ bounds) {
    const uint64_t id = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= (uint64_t)n_src * nb1) return;
    const uint32_t s = (uint32_t)(id / nb1), j = (uint32_t)(id % nb1);
    const unsigned long long n = src_count[s];
    const uint64_t bb = (uint64_t)b_begin + j;
    unsigned long long lo = 0, hi = n;
    if (bb >= (1ULL << bucket_bits)) lo = n;
    else {
        const unsigned long long target = bb << (64 - bucket_bits);
        const unsigned long long* src = parts + src_off[s];
        const uint32_t width = src_width[s];
        while (lo < hi) {
            const unsigned long long mid = (lo + hi) >> 1;
            if (src[mid * width] < target) lo = mid + 1; else hi = mid;
        }
    }
    bounds[id] = lo;
}

// Emission.  Slots are handled in chunks of kAggThreads consecutive slots, lane = slot: shared-memory accesses are
// conflict-free, the inversion walks of neighbouring lanes touch neighbouring slots, and the columns leave in
// (almost) consecutive order.
// Pass A: kept flags; kept slots per (chunk, warp) in s_wc.  Returns this thread's occupied count.
constexpr int kAggMaxChunks = (kAggMaxSlots + kMaxProbe + kAggThreads - 1) / kAggThreads;
static_assert(kAggMaxChunks * (kAggThreads / 32) <= kAggThreads, "the scan of the per-(chunk, warp) counts takes one value per thread");
template <int MODE>
__device__ __forceinline__ uint32_t agg_mark(const AggParams2& p, const AggTable& t, uint32_t* s_wc) {
    uint32_t occ = 0;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t c = 0;
    for (uint32_t i0 = 0; i0 < t.total; i0 += kAggThreads, ++c) {
        const uint32_t i = i0 + threadIdx.x;
        uint32_t kf = 0;
        if (i < t.total && t.keys[i] != kEmptyKey) {
            occ++;
            if (MODE == 6 || MODE == 7) {
                for (uint32_t r = 0; r < p.round_rows; ++r) kf |= t.w32[r * t.total + i] >= p.min_abundance;
            } else if (MODE == 5 || p.keep_singletons) kf = 1;
            else if (MODE == 3) {
                uint32_t pc = 0;
                for (uint32_t s = 0; s < p.n_src; ++s) {
                    const uint32_t e = t.w32[s * t.total + i];
                    if (e) {
                        const unsigned long long* ent = p.parts + p.src_off[s] + (unsigned long long)(e - 1u) * (1u + p.src_words[s]);
                        for (uint32_t w = 0; w < p.src_words[s]; ++w) pc += __popcll(ent[1 + w]);
                    }
                }
                kf = pc >= 2;
            } else {
                uint32_t pc = 0;
                for (uint32_t h = 0; h < 2 * p.n_words; ++h) pc += __popc(t.w32[h * t.total + i]);
                kf = pc >= 2;
            }
        }
        if (i < t.total) t.kept[i] = (uint8_t)(kf << 7);        // bit 7 = kept, bits 0-6 = the rank correction of agg_fix
        const uint32_t bal = __ballot_sync(0xffffffffu, kf != 0);
        if (lane == 0) s_wc[c * (kAggThreads / 32) + warp] = (uint32_t)__popc(bal);
    }
    return occ;
}

// Rank of a kept slot = kept slots before it, corrected by the inversions it takes part in.  The home slot is monotone
// in the key and probing never wraps, so a LATER slot i can only be out of order with the slots [home(key_i), i): a
// larger key at j < i has home(key_j) >= home(key_i) and sits at or after its home.  Every inversion is therefore found
// by its later element with a walk as long as that element's displacement (0.5 slots on average at half load, instead
// of the whole cluster in both directions).
// Pass B1: the later element of an inversion adds one to the earlier element's correction (bits 0-6 of its flag byte;
// at most kMaxProbe - 1 = 95 later slots can reach back to a slot, so the counter never touches bit 7).
__device__ __forceinline__ void agg_fix(const AggTable& t, uint32_t shift) {
    uint32_t* const kept32 = reinterpret_cast<uint32_t*>(t.kept);
    for (uint32_t i = threadIdx.x; i < t.total; i += kAggThreads) {
        if (!(t.kept[i] & 0x80u)) continue;
        const unsigned long long key = t.keys[i];
        uint32_t dec = 0;
        for (uint32_t j = home_slot(key, shift, t.slots); j < i; ++j)
            if (t.keys[j] > key && (t.kept[j] & 0x80u)) { atomicAdd(&kept32[j >> 2], 1u << (8u * (j & 3u))); ++dec; }
        t.dec[i] = (uint8_t)dec;             // the emission does not walk again
    }
}

// Pass B2: emission at out[base + rank], rank = kept slots before + correction - own inversions.  s_wp = exclusive scan of s_wc.
template <int MODE>
__device__ __forceinline__ void agg_emit(const AggParams2& p, const AggTable& t, const uint32_t* s_wp,
                                         unsigned long long base, uint32_t b, uint32_t key_bits, uint32_t shift) {
    const unsigned long long key_mask = (1ULL << key_bits) - 1;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t c = 0;
    for (uint32_t i0 = 0; i0 < t.total; i0 += kAggThreads, ++c) {
        const uint32_t i = i0 + threadIdx.x;
        const uint32_t flag = i < t.total ? t.kept[i] : 0u;
        const bool kf = (flag & 0x80u) != 0;
        const uint32_t bal = __ballot_sync(0xffffffffu, kf);
        if (!kf) continue;
        const unsigned long long key = t.keys[i];
        const uint32_t rank = s_wp[c * (kAggThreads / 32) + warp] + (uint32_t)__popc(bal & ((1u << lane) - 1u)) + (flag & 0x7Fu) - t.dec[i];
        const unsigned long long o = base + rank;
        if (o < p.cap) {
            const unsigned long long h = ((unsigned long long)b << key_bits) | (key & key_mask);
            if (MODE == 6) {
                unsigned long long bits = 0;
                for (uint32_t r = 0; r < p.round_rows; ++r)
                    if (t.w32[r * t.total + i] >= p.min_abundance) bits |= 1ULL << (63u - ((p.round_row0 + r) & 63u));
                p.out_wide[o] = make_ulonglong2((h << p.out_wbits) | p.out_word, bits);
                continue;
            }
            p.out_keys[o] = (MODE == 5 || (MODE == 3 && p.partial_out)) ? h : kunhash(h);
            if (MODE == 3) {
                // The words come from the sources' entries (random 16 / 24 / 40-byte reads out of L2).  Four sources at a
                // time: all their references first, then all the loads, then the stores -- one dependent load at a time left
                // the kernel waiting on the scoreboard for a third of its samples (profiles/r02_merge_emit.txt: aggregate 1.05 ->
                // 0.88 ms at 8 sources x 2 words; a variant that walked the word rows through a (source, word) table in
                // shared memory, eight at a time, took 1.00 ms).
                unsigned long long* const orow = p.out_words + o;
                for (uint32_t s0 = 0; s0 < p.n_src; s0 += 4) {
                    uint32_t e[4];
                    unsigned long long v0[4], v1[4];
                    const unsigned long long* ent[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) e[q] = s0 + q < p.n_src ? t.w32[(s0 + q) * t.total + i] : 0u;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        v0[q] = v1[q] = 0ULL;
                        ent[q] = nullptr;
                        if (e[q]) {
                            const uint32_t nw = p.src_words[s0 + q];
                            ent[q] = p.parts + p.src_off[s0 + q] + (unsigned long long)(e[q] - 1u) * (1u + nw);
                            if (nw >= 1) v0[q] = __ldg(ent[q] + 1);
                            if (nw >= 2) v1[q] = __ldg(ent[q] + 2);
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        if (s0 + q >= p.n_src) break;
                        const uint32_t nw = p.src_words[s0 + q], wo = p.src_woff[s0 + q];
                        if (nw >= 1) orow[(unsigned long long)wo * p.cap] = v0[q];
                        if (nw >= 2) orow[(unsigned long long)(wo + 1) * p.cap] = v1[q];
                        for (uint32_t w0 = 2; w0 < nw; w0 += 4) {      // (sources of more than 128 genomes: four more words at a time)
                            unsigned long long x[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) x[j] = (ent[q] && w0 + j < nw) ? __ldg(ent[q] + 1 + w0 + j) : 0ULL;
#pragma unroll
                            for (int j = 0; j < 4; ++j) if (w0 + j < nw) orow[(unsigned long long)(wo + w0 + j) * p.cap] = x[j];
                        }
                    }
                }
            } else {
                for (uint32_t w = 0; w < p.n_words; ++w) {
                    p.out_words[w * p.cap + o] = ((unsigned long long)t.w32[(2 * w + 1) * t.total + i] << 32) | t.w32[2 * w * t.total + i];
                }
            }
        }
    }
}

// Ordered emission: where does (virtual) bucket idx start?  Called by the whole first warp.  The bucket publishes its own
// count, sums its predecessors' words 32 at a time until one of them carries an inclusive prefix, then publishes its
// own inclusive prefix.  The words are self-validating (flag bits + value in one 64-bit store), so relaxed accesses do;
// buckets are dealt by ticket, so every predecessor belongs to a CTA that is already running (no deadlock whatever
// the residency).
constexpr unsigned long long kAggPubInc = 1ULL << 63, kAggPubOwn = 1ULL << 62, kAggPubMask = (1ULL << 62) - 1;
__device__ __forceinline__ unsigned long long agg_reserve_ordered(const AggParams2& p, uint32_t idx, unsigned long long total) {
    const uint32_t lane = threadIdx.x & 31u;
    if (lane == 0) {
        atomicAdd(&p.scalars[S_U_NEEDED], total);
        st_relaxed_u64(p.pub + idx, (idx == 0 ? kAggPubInc : kAggPubOwn) | total);
    }
    if (idx == 0) return 0;
    unsigned long long excl = 0;
    for (long long j = (long long)idx - 1;; j -= 32) {
        const long long q = j - (long long)lane;
        unsigned long long v;
        do { v = q >= 0 ? ld_relaxed_u64(p.pub + q) : kAggPubInc; } while (!__all_sync(0xffffffffu, (v >> 62) != 0));
        const uint32_t inc = __ballot_sync(0xffffffffu, (v & kAggPubInc) != 0);
        unsigned long long val = v & kAggPubMask;
        if (inc && lane > (uint32_t)(__ffs(inc) - 1)) val = 0;
#pragma unroll
        for (int o = 16; o; o >>= 1) val += __shfl_xor_sync(0xffffffffu, val, o);
        excl += val;
        if (inc) break;
    }
    if (lane == 0) st_relaxed_u64(p.pub + idx, kAggPubInc | (excl + total));
    return excl;
}

template <int MODE>
__global__ void __launch_bounds__(kAggThreads, kAggCtasPerSm)
k_aggregate_cols(const AggParams2 p) {
    extern __shared__ unsigned long long s_tab[];
    __shared__ uint32_t s_overflow, s_sp;
    __shared__ uint32_t s_depth[72];
    __shared__ unsigned long long s_idx[72];
    __shared__ uint32_t s_warp[33];
    __shared__ unsigned long long s_base;
    AggTable t;
    t.slots = p.slots; t.total = p.slots + kMaxProbe;
    t.keys = s_tab;
    t.w32 = reinterpret_cast<uint32_t*>(s_tab + t.total);
    t.kept = reinterpret_cast<uint8_t*>(t.w32 + (size_t)p.table_u32 * t.total);
    t.dec = t.kept + ((t.total + 3u) & ~3u);
    const uint32_t key_bits = 64 - p.bucket_bits;
    const uint32_t n_chunks = (t.total + kAggThreads - 1) / kAggThreads;     // <= kAggMaxChunks (slots <= 16384)
    __shared__ uint32_t s_wc[kAggMaxChunks * (kAggThreads / 32)];

    // A virtual bucket = bucket b restricted to the key sub-range `sub` of 2^sub_bits: the scatter can then use
    // 2^sub_bits fewer buckets (longer runs per tile) than the table size demands.  The CTAs of one bucket's
    // sub-ranges have adjacent block indices, run at the same time and share the bucket's records through L2.
    const uint32_t sb = p.sub_bits;
    const uint32_t vb_base = p.b_begin << sb;
    __shared__ uint32_t s_vb;
    for (uint32_t it = 0;; ++it) {
        uint32_t vb = vb_base + blockIdx.x + it * gridDim.x;
        if (p.ordered) {
            __syncthreads();
            if (threadIdx.x == 0) s_vb = atomicAdd(p.ticket, 1u);
            __syncthreads();
            vb = vb_base + s_vb;
        }
        if (vb >= (p.b_end << sb)) break;
        const uint32_t b = vb >> sb, sub = vb & ((1u << sb) - 1u);
        uint32_t n = 0;
        const unsigned long long* recs = nullptr;
        if (MODE == 3) {
            const uint32_t nb1 = p.b_end - p.b_begin + 1;
            for (uint32_t s = 0; s < p.n_src; ++s)
                n += (uint32_t)(p.bounds[(size_t)s * nb1 + (b - p.b_begin) + 1] - p.bounds[(size_t)s * nb1 + (b - p.b_begin)]);
        } else {
            const unsigned long long rbeg = p.begin[b], rend = p.end[b];
            n = rbeg < rend ? (uint32_t)(rend - rbeg) : 0u;
            recs = p.records + (MODE >= 4 ? (unsigned long long)p.wide_stride * rbeg : rbeg);
        }
        if (n == 0) {
            if (threadIdx.x == 0) { p.bucket_base[vb - vb_base] = 0; p.bucket_count[vb - vb_base] = 0; }
            // an empty bucket only publishes its (zero) count: its successors look past it
            if (p.ordered && threadIdx.x == 0) st_relaxed_u64(p.pub + (vb - vb_base), (vb == vb_base ? kAggPubInc : kAggPubOwn));
            continue;
        }
        // phase 0: the whole (virtual) bucket in one table; on overflow phase 1 counts over its key sub-ranges and
        // phase 2 emits them in ascending order
        uint32_t phase = 0;
        uint32_t bucket_total = 0, emitted = 0, bucket_occ = 0, splits = 0;
        __syncthreads();
        if (threadIdx.x == 0) { s_sp = 1; s_depth[0] = sb; s_idx[0] = sub; }
        while (true) {
            __syncthreads();
            if (s_sp == 0) {
                if (phase != 1) break;
                __syncthreads();          // everyone has seen the empty stack before it is refilled
                // counting sweep done: reserve the bucket's chunk, then emit
                if (p.ordered) {
                    if (threadIdx.x < 32) {
                        const unsigned long long base = agg_reserve_ordered(p, vb - vb_base, bucket_total);
                        if (threadIdx.x == 0) s_base = base;
                    }
                } else if (threadIdx.x == 0) s_base = atomicAdd(&p.scalars[S_U_NEEDED], (unsigned long long)bucket_total);
                if (threadIdx.x == 0) {
                    s_sp = 0;
                    s_depth[s_sp] = sb + 1; s_idx[s_sp] = 2ULL * sub + 1; s_sp++;
                    s_depth[s_sp] = sb + 1; s_idx[s_sp] = 2ULL * sub; s_sp++;
                }
                phase = 2;
                continue;
            }
            const uint32_t depth = s_depth[s_sp - 1];
            const unsigned long long ridx = s_idx[s_sp - 1];
            __syncthreads();
            if (threadIdx.x == 0) { s_sp--; s_overflow = 0; }
            for (uint32_t i = threadIdx.x; i < t.total; i += kAggThreads) t.keys[i] = kEmptyKey;
            for (uint32_t i = threadIdx.x; i < t.total * (p.table_u32 / 2); i += kAggThreads) reinterpret_cast<unsigned long long*>(t.w32)[i] = 0;
            __syncthreads();
            if (MODE == 3) {
                if (depth == 0) agg_stream_parts<false>(p, t, b, key_bits, 0, 0, &s_overflow);
                else agg_stream_parts<true>(p, t, b, key_bits, depth, ridx, &s_overflow);
            } else {
                if (depth == 0) agg_stream_wide<false, (MODE >= 6)>(p, t, recs, n, key_bits, 0, 0, &s_overflow);
                else agg_stream_wide<true, (MODE >= 6)>(p, t, recs, n, key_bits, depth, ridx, &s_overflow);
            }
            __syncthreads();
            if (s_overflow) {
                // split this key range in two, lower half first (terminates: a range of one key needs one slot)
                if (threadIdx.x == 0) {
                    if (phase == 0) {
                        s_depth[s_sp] = sb + 1; s_idx[s_sp] = 2ULL * sub + 1; s_sp++;
                        s_depth[s_sp] = sb + 1; s_idx[s_sp] = 2ULL * sub; s_sp++;
                    } else {
                        s_depth[s_sp] = depth + 1; s_idx[s_sp] = ridx * 2 + 1; s_sp++;
                        s_depth[s_sp] = depth + 1; s_idx[s_sp] = ridx * 2; s_sp++;
                    }
                }
                if (phase == 0) phase = 1;
                if (phase == 1) splits++;
                continue;
            }
            const uint32_t occ = agg_mark<MODE>(p, t, s_wc);
            __syncthreads();
            uint32_t total_kept, total_occ;
            {
                constexpr uint32_t kWarps = kAggThreads / 32;
                const uint32_t v = threadIdx.x < n_chunks * kWarps ? s_wc[threadIdx.x] : 0u;
                const uint32_t e = block_excl_scan<kAggThreads>(v, s_warp, total_kept);
                if (threadIdx.x < n_chunks * kWarps) s_wc[threadIdx.x] = e;
            }
            if (phase != 2) { block_excl_scan<kAggThreads>(occ, s_warp, total_occ); bucket_occ += total_occ; }
            if (phase == 1) { bucket_total += total_kept; continue; }
            if (phase == 0) {
                bucket_total = total_kept;
                if (p.ordered) {
                    if (threadIdx.x < 32) {
                        const unsigned long long base = agg_reserve_ordered(p, vb - vb_base, total_kept);
                        if (threadIdx.x == 0) s_base = base;
                    }
                } else if (threadIdx.x == 0) s_base = atomicAdd(&p.scalars[S_U_NEEDED], (unsigned long long)total_kept);
            }
            agg_fix(t, 64 - key_bits + depth);
            __syncthreads();
            agg_emit<MODE>(p, t, s_wc, s_base + emitted, b, key_bits, 64 - key_bits + depth);
            emitted += total_kept;
        }
        if (threadIdx.x == 0) {
            p.bucket_base[vb - vb_base] = s_base;
            p.bucket_count[vb - vb_base] = bucket_total;
            atomicAdd(&p.scalars[S_N_DISTINCT], (unsigned long long)bucket_occ);
            if (splits) atomicAdd(&p.scalars[S_N_SPLITS], (unsigned long long)splits);
        }
    }
}

// bucket chunks (arbitrary order in tmp) -> final arrays in bucket order: one CTA per bucket
__global__ void __launch_bounds__(256)
k_gather_buckets(const unsigned long long* __restrict__ tmp_keys, const unsigned long long* __restrict__ tmp_words,
                 unsigned long long tmp_cap, const unsigned long long* __restrict__ bucket_base,
                 const unsigned long long* __restrict__ offsets, uint32_t B, uint32_t W, unsigned long long U,
                 unsigned long long* __restrict__ keys, unsigned long long* __restrict__ words, unsigned long long out_stride) {
    for (uint32_t b = blockIdx.x; b < B; b += gridDim.x) {
        const unsigned long long src = bucket_base[b], dst = offsets[b], n = offsets[b + 1] - dst;
        for (unsigned long long i = threadIdx.x; i < n; i += blockDim.x) {
            keys[dst + i] = tmp_keys[src + i];
            for (uint32_t w = 0; w < W; ++w) words[(unsigned long long)w * out_stride + dst + i] = tmp_words[(unsigned long long)w * tmp_cap + src + i];
        }
    }
    (void)U;
}

// abundance builds: the solid presence records of all rounds (16 bytes each; a round leaves one chunk per virtual
// bucket) -> bucket-contiguous order for the final presence aggregate.  segs = [source, destination, count] triples.
__global__ void __launch_bounds__(128)
k_gather_segments(const ulonglong2* __restrict__ src, const unsigned long long* __restrict__ segs, uint32_t n_segs,
                  ulonglong2* __restrict__ dst) {
    for (uint32_t s = blockIdx.x; s < n_segs; s += gridDim.x) {
        const unsigned long long a = segs[3 * (size_t)s], d = segs[3 * (size_t)s + 1], n = segs[3 * (size_t)s + 2];
        for (unsigned long long i = threadIdx.x; i < n; i += blockDim.x) dst[d + i] = __ldcs(src + a + i);
    }
}

// ------------------------------------------------------------------------------------------
// multi-GPU: partial columns out (AoS records for the all-to-all) and owner-side partition
// ------------------------------------------------------------------------------------------
// record i = [hash, word_0 .. word_{W-1}]
// The same gather, fused with the all-to-all: owner d's slice (buckets [first[d], first[d + 1])) is stored straight into
// rank d's receive buffer over NVLink (peer pointers from torch symmetric memory), at the word offset the counts
// exchange assigned to this rank.  No send buffer, no NCCL send / recv; the ranks meet at one barrier afterwards.
struct PeerSlices {
    unsigned long long* dst[16];          // peer d's receive buffer + this rank's word offset in it
    uint32_t first[17];                   // first (virtual) bucket of owner d; first[n] = B
    uint32_t n;
    uint32_t rot;                         // the walk over the buckets starts here (the first bucket of the NEXT rank's range)
};
__global__ void __launch_bounds__(256)
k_gather_buckets_peers(const unsigned long long* __restrict__ tmp_keys, const unsigned long long* __restrict__ tmp_words,
                       unsigned long long tmp_cap, const unsigned long long* __restrict__ bucket_base,
                       const unsigned long long* __restrict__ offsets, uint32_t B, uint32_t W, const PeerSlices ps) {
    // Every rank starts with the buckets of the rank after it and ends with its own: at any moment the P exporters store
    // into P different receivers.  Walked from bucket 0 on every rank, all of them filled owners 0 .. 4 first and 5 .. 7
    // afterwards -- an all-to-all in which five, then three receivers take everybody's stores (N = 8: 0.57 ms for 214 MB
    // per rank over NVLink).
    for (uint32_t i = blockIdx.x; i < B; i += gridDim.x) {
        uint32_t b = i + ps.rot;
        if (b >= B) b -= B;
        uint32_t d = 0;
        while (d + 1 < ps.n && b >= ps.first[d + 1]) ++d;
        const unsigned long long src = bucket_base[b], d0 = offsets[b] - offsets[ps.first[d]], n = offsets[b + 1] - offsets[b];
        unsigned long long* __restrict__ dst = ps.dst[d] + d0 * (1 + W);
        // (a bucket's chunk is far below 2^32 cells: 32-bit index arithmetic, the 64-bit division per cell was most of the
        // kernel's instructions)
        const uint32_t width = 1u + W, cells = (uint32_t)n * width;
        const unsigned long long* __restrict__ keys = tmp_keys + src;
        const unsigned long long* __restrict__ words = tmp_words + src;
        // four cells per thread and step, the loads ahead of the stores: with one 8-byte load in flight per thread the kernel
        // ran at 1.9 TB/s of combined traffic (0.25 ms for 240 MB on two GPUs), bound by latency, not by HBM or NVLink
        for (uint32_t c0 = threadIdx.x; c0 < cells; c0 += 4 * blockDim.x) {
            unsigned long long v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t c = c0 + q * blockDim.x;
                if (c < cells) {
                    const uint32_t i = c / width, f = c - i * width;
                    v[q] = f == 0 ? keys[i] : words[(unsigned long long)(f - 1) * tmp_cap + i];
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t c = c0 + q * blockDim.x;
                if (c < cells) dst[c] = v[q];
            }
        }
    }
}

// bucket chunks (completion order) -> AoS records [hash, word_0 .. word_{W-1}] in bucket order: the gather and the
// export of a partial build in one pass
__global__ void __launch_bounds__(256)
k_gather_buckets_aos(const unsigned long long* __restrict__ tmp_keys, const unsigned long long* __restrict__ tmp_words,
                     unsigned long long tmp_cap, const unsigned long long* __restrict__ bucket_base,
                     const unsigned long long* __restrict__ offsets, uint32_t B, uint32_t W, unsigned long long* __restrict__ dst) {
    for (uint32_t b = blockIdx.x; b < B; b += gridDim.x) {
        const unsigned long long src = bucket_base[b], d0 = offsets[b], n = offsets[b + 1] - d0;
        // one u64 of the AoS output per thread and step: coalesced stores, the loads hit W + 1 runs
        const uint32_t width = 1u + W, cells = (uint32_t)n * width;      // (32-bit index arithmetic: see k_gather_buckets_peers)
        const unsigned long long* __restrict__ keys = tmp_keys + src;
        const unsigned long long* __restrict__ words = tmp_words + src;
        unsigned long long* __restrict__ out = dst + d0 * width;
        for (uint32_t c0 = threadIdx.x; c0 < cells; c0 += 4 * blockDim.x) {      // (four loads in flight per thread)
            unsigned long long v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t c = c0 + q * blockDim.x;
                if (c < cells) {
                    const uint32_t i = c / width, f = c - i * width;
                    v[q] = f == 0 ? keys[i] : words[(unsigned long long)(f - 1) * tmp_cap + i];
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t c = c0 + q * blockDim.x;
                if (c < cells) out[c] = v[q];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// emit
// ------------------------------------------------------------------------------------------
__global__ void k_kmer_strings(const unsigned long long* __restrict__ kmers, uint64_t j0, uint64_t n_bytes,
                               uint32_t k, char* __restrict__ dst) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bytes) return;
    const uint64_t j = i / k; const uint32_t c = (uint32_t)(i % k);
    const uint32_t code = (uint32_t)(kmers[j0 + j] >> (2 * (k - 1 - c))) & 3u;
    dst[i] = "ACTG"[code];
}

// rows [j0, j0 + n_rows) of the TSV body; row width = k + 2G + 1
__global__ void k_format_tsv(const unsigned long long* __restrict__ kmers, const unsigned long long* __restrict__ matrix,
                             uint64_t pitch, uint32_t G, uint32_t k, uint64_t j0, uint64_t n_bytes, char* __restrict__ dst) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_bytes) return;
    const uint32_t roww = k + 2 * G + 1;
    const uint64_t j = j0 + i / roww; const uint32_t c = (uint32_t)(i % roww);
    char out;
    if (c < k) out = "ACTG"[(uint32_t)(kmers[j] >> (2 * (k - 1 - c))) & 3u];
    else if (c == roww - 1) out = '\n';
    else if (((c - k) & 1u) == 0) out = '\t';
    else {
        const uint32_t g = (c - k) >> 1;
        out = ((matrix[(uint64_t)(g >> 6) * pitch + j] >> (63 - (g & 63))) & 1ULL) ? '1' : '0';
    }
    dst[i] = out;
}

}  // namespace grmkm
