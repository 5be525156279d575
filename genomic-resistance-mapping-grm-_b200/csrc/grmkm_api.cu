// grmkm_api.cu -- C ABI (include/grmkm.h) and host orchestration of the sm_100a kernels.
// One context = one GPU.  No CPU fallback: without a device grmkm_create fails.
#include "../../include/grmkm.h"
#include "grmkm_kernels.cuh"
#include "grmkm_units.cuh"
#include "grmkm_result.cuh"
#include "grmkm_synth.cuh"
#include "grmkm_scm.cuh"
#include "grmkm_cart.cuh"
#include "grmkm_query.cuh"
#include "grmkm_eval.cuh"
#include "grmkm_shard.cuh"
#include "grmkm_patterns.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <nvtx3/nvToolsExt.h>      // header-only; the ranges cost nothing until a tool (nsys, ncu --nvtx) attaches
#include <zlib.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>

using namespace grmkm;

namespace {

thread_local std::string g_create_error;

// NVTX range on the calling host thread: the stages of a build as a profiler sees them enqueued
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { end(); }
    void end() { if (open) { nvtxRangePop(); open = false; } }      // ranges are closed in the order they were opened
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
    bool open = true;
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct Input {
    uint32_t row = 0;
    uint32_t kind = 0;
    const uint8_t* host = nullptr;
    const uint8_t* dev = nullptr;
    uint64_t len = 0;
    std::vector<uint8_t> owned;
};

constexpr uint32_t kMaxGenomes = 32768;
constexpr uint64_t kBatchBytes = 32ull << 20;      // text per pipelined H2D batch (GRMKM_BATCH_BYTES overrides, for tests)

// H2D gate.  Several contexts of one device may build at the same time (builder.BuildPipeline: a series of datasets,
// one worker thread per context).  Their host->device legs follow one another instead of sharing the link: the first
// copy of a build waits for the event the previous build recorded behind its last copy, so the builds fall into
// step -- one copies its text in while the other runs its dedupe / expand / aggregate kernels and copies its result
// out (PCIe is full duplex).  With one context the event is long complete and the wait costs nothing.
struct H2dGate {
    std::mutex mu;                    // held while a build enqueues its copies: the order of the legs = the order of the locks
    cudaEvent_t done[64] = {};        // per device, created on first use, never destroyed (process lifetime)
};
H2dGate g_h2d;

enum Stage { T_START = 0, T_H2D, T_PARSE, T_PACK, T_COUNT, T_BOUNDS, T_SCATTER, T_ABUND, T_DEDUPE, T_EXPAND, T_AGG, T_SORT, T_N };

}  // namespace

struct grmkm_ctx {
    grmkm_config cfg{};
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    std::vector<Input> inputs;
    uint32_t n_genomes_decl = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    void* h_tab = nullptr;         // page-locked arena for the per-batch host tables (files, stream starts, ticket order)
    size_t h_tab_cap = 0, h_tab_used = 0;
    uint64_t wide_hint = 0;
    // the packed stream and the tile words of the NEXT build are cleared on a side stream while this build's dedupe /
    // expand / aggregate run (they are dead once the scatter has consumed them)
    cudaStream_t aux_stream = nullptr;
    cudaEvent_t ev_scattered = nullptr, ev_cleared = nullptr;
    bool pre_pending = false;
    const void *pre_codes = nullptr, *pre_valid = nullptr, *pre_pub = nullptr;
    uint64_t pre_groups = 0, pre_pub_bytes = 0;
    uint64_t pass_groups = 0, pass_pub_bytes = 0;
    uint64_t wide_capped_need = 0;   // an expansion-buffer request of up to this many bytes was capped by free memory
    uint64_t ucap_hint = 0;        // columns of the previous build + headroom (sizes the aggregate's output)        // wide records of the previous build (sizes the expansion's bucket regions)

    // device buffers (grow-only, reused across builds)
    DevBuf in, files, hdr0, tile_file, tile_pub, tile_order, fss, codes, valid, hist,
        offsets, offsets2, bcounts, ukeys, uwords, kmers, matrix,
        scalars, fmt, synth, refs, stile_file, bbase, apub, masks, units, ucur, ubeg, wu, wide,
        racc,            // abundance builds: the solid presence records of the rounds done so far
        aux,             // result-side kernels: row mask / per-column sums / checksum / bit rows / Gram matrix
        scm,             // grmkm_scm_run: masks, bests, blacklist bits, per-CTA bests, selections
        scm_list,        // grmkm_scm_run: the tie list and the statistics of its rules
        cart,            // grmkm_cart_run: per-level node arguments, bests, tie totals, per-CTA bests and tie counts, splits
        cart_bl,         // grmkm_cart_run: blacklist bits (one per k-mer)
        cart_masks[2],   // grmkm_cart_run: P and N of the open nodes of this level / of the next level
        cart_list,       // grmkm_cart_run: the tie list
        qry,             // grmkm_query: key table, slot -> key index, caller column -> key index, totals
        qplane,          // grmkm_query: presence plane or counters of one row range
        qout,            // grmkm_query: one row range's word rows in the caller's column order
        eval,            // grmkm_eval_run: job arguments, rules, nodes, example masks, counts
        shard_idx,       // sharded runs: the local indices of the columns this rank sends, and their packed words
        shard_cols,      // sharded runs: the compact matrix of the exchanged columns
        pat,             // grmkm_patterns (source side): fingerprints, grouping table, ids, members, sort scratch
        pat_mult;        // a pattern matrix (grmkm_patterns' destination): every column's multiplicity, uint32
    cudaEvent_t ev_query[2] = {nullptr, nullptr};   // grmkm_query: device time of the call
    uint64_t racc_hint = 0;        // records of the previous abundance build + headroom
    std::vector<uint64_t> merge_h_off;   // row-block merge of a partial build: chunk offsets of the merge buckets
    uint32_t merge_bits = 0;
    uint64_t merge_cap = 0;
    size_t device_bytes = 0;

    cudaEvent_t ev[T_N]{};
    bool ev_ok = false;

    // H2D pipeline: copy stream, "batch copied" / "staging half free" events
    uint64_t batch_bytes = kBatchBytes;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2]{}, ev_free[2]{};

    // page-locked host copy of the result (grmkm_host_result)
    void* host_res = nullptr;
    size_t host_res_cap = 0;

    // result
    bool built = false;
    uint64_t U = 0;
    uint64_t pitch = 0;            // u64 words between two word rows of `matrix` (>= U: the ordered emission writes every row at
                                   // the stride of its capacity guess, because U is only known when the last bucket is done)
    uint32_t W = 0, G = 0;
    bool slice = false;            // the result is one owner's slice of a multi-GPU merge (grmkm_merge_partials, n_ranks > 1)
    bool pat_mult_on = false;      // the result is a pattern matrix whose pat_mult holds its columns' multiplicities
    grmkm_stats stats{};
    grmkm_times times{};

    // multi-GPU partial state
    uint32_t part_ranks = 0;
    std::vector<uint64_t> part_counts;
    uint64_t part_total = 0, part_cap = 0;      // partial columns of the last partial build; stride of its bucket chunks
    uint32_t part_buckets = 0;
    uint32_t part_words = 0;
    uint32_t cur_bucket_bits = 0;
    int32_t xrank = -1;                  // this context's rank in the exchange (grmkm_set_exchange_rank); -1: the device index

    // grmkm_scm_run results: per fit, its steps and their equivalent rules
    std::vector<std::vector<grmkm_scm_step>> scm_steps;
    std::vector<std::vector<uint64_t>> scm_equiv;
    // grmkm_cart_run results: per tree, its nodes and their recorded equivalent rules
    std::vector<std::vector<grmkm_cart_node>> cart_nodes;
    std::vector<std::vector<uint64_t>> cart_equiv;
};

namespace {

int fail(grmkm_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}

#define CU_TRY(c, call)                                                                                   \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess)                                                                            \
            return fail((c), GRMKM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));           \
    } while (0)

int ensure(grmkm_ctx* c, DevBuf& b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b.cap >= bytes) return GRMKM_OK;
    if (b.p) { cudaFree(b.p); c->device_bytes -= b.cap; b.p = nullptr; b.cap = 0; }
    size_t want = (bytes + 255) & ~size_t(255);
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        b.p = nullptr;
        return fail(c, GRMKM_E_NOMEM, "cudaMalloc of " + std::to_string(want) + " bytes failed: " + cudaGetErrorString(e));
    }
    b.cap = want;
    c->device_bytes += want;
    return GRMKM_OK;
}
#define ENSURE(c, buf, bytes) do { int r_ = ensure((c), (buf), (bytes)); if (r_) return r_; } while (0)

void release(grmkm_ctx* c, DevBuf& b) {
    if (b.p) { cudaFree(b.p); c->device_bytes -= b.cap; }
    b.p = nullptr; b.cap = 0;
}

uint32_t ceil_log2(uint64_t x) {
    uint32_t b = 0;
    while ((1ULL << b) < x) ++b;
    return b;
}

struct Launches { uint32_t n = 0; };

int read_file(grmkm_ctx* c, const char* path, std::vector<uint8_t>& out) {
    const size_t L = strlen(path);
    const bool gz = L > 3 && strcmp(path + L - 3, ".gz") == 0;
    if (gz) {
        gzFile f = gzopen(path, "rb");
        if (!f) return fail(c, GRMKM_E_IO, std::string("cannot open ") + path);
        gzbuffer(f, 1 << 20);
        std::vector<uint8_t> buf(1 << 22);
        int n;
        while ((n = gzread(f, buf.data(), (unsigned)buf.size())) > 0) out.insert(out.end(), buf.begin(), buf.begin() + n);
        const bool bad = n < 0;
        gzclose(f);
        if (bad) return fail(c, GRMKM_E_IO, std::string("cannot inflate ") + path);
        return GRMKM_OK;
    }
    FILE* f = fopen(path, "rb");
    if (!f) return fail(c, GRMKM_E_IO, std::string("cannot open ") + path);
    fseek(f, 0, SEEK_END);
    long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    if (sz < 0) { fclose(f); return fail(c, GRMKM_E_IO, std::string("cannot size ") + path); }
    out.resize((size_t)sz);
    size_t got = sz ? fread(out.data(), 1, (size_t)sz, f) : 0;
    fclose(f);
    if (got != (size_t)sz) return fail(c, GRMKM_E_IO, std::string("short read on ") + path);
    return GRMKM_OK;
}

size_t agg_smem_budget(const grmkm_ctx* c) {
    // leave room for the kernel's static shared memory
    size_t lim = c->smem_optin ? c->smem_optin : 227 * 1024;
    lim = (lim + 1024) / kAggCtasPerSm - 1024;       // every resident CTA also costs 1 KB of system shared memory
    return lim - 4096;      // static shared memory of k_aggregate_cols: 3.2 KB
}

// table = (slots + kMaxProbe) x (u64 key + `cells` u32 cells + u8 kept flag / correction + u8 own inversions); slots = home
// positions.  cells = 2 W presence half-words (presence builds), one counter per genome row of the round rounded up to
// even (abundance rounds), one entry reference per source (owner-side merge).
uint32_t table_slots(const grmkm_ctx* c, uint32_t cells) {
    const size_t budget = agg_smem_budget(c);
    const size_t total = (budget - 8) / (10 + 4 * (size_t)cells);
    if (total < (size_t)kMaxProbe + 256) return 0;
    return (uint32_t)std::min<size_t>(kAggMaxSlots, total - kMaxProbe);
}
size_t table_smem(uint32_t slots, uint32_t cells) {
    return (((size_t)slots + kMaxProbe) * (10 + 4 * (size_t)cells) + 8 + 15) & ~size_t(15);
}

constexpr uint32_t kUnitMaxBucketBits = 11;      // the unit expansion sorts tiles over at most 2^11 hash buckets
constexpr uint32_t kMaxSubBits = 3;              // key sub-ranges (virtual buckets) per bucket: up to 2^3
constexpr uint32_t kRoundMaxRows = 4;            // genome rows per abundance round (one u32 counter plane each)
constexpr uint32_t kBlockRows = 256;             // presence builds of more genomes than this run in row blocks (build_row_blocks)

bool abundance_build(const grmkm_ctx* c) { return c->cfg.min_abundance > 1 || (c->cfg.flags & GRMKM_FLAG_COUNTS); }

// ---- abundance rounds: the genomes of a -abundance-min > 1 build are counted a few rows at a time (the counters of a
// round live in the shared-memory tables, and the distinct k-mers of read sets are mostly sequencing errors that are
// unique to their genome).  A round holds consecutive rows of ONE 64-row matrix word, at most kRoundMaxRows of them,
// and as much text as the tables of one pass hold (estimated: one distinct k-mer per 10 bytes of text).
struct Round { uint32_t f0, f1, row0, n_rows; uint64_t bytes; };

std::vector<Round> plan_rounds(const grmkm_ctx* c, uint32_t G, const std::vector<uint32_t>& first_file /* [G + 1] */,
                               const std::vector<uint64_t>& row_bytes) {
    std::vector<Round> rounds;
    if (c->cfg.flags & GRMKM_FLAG_COUNTS) {          // pooled count table: everything is one row
        rounds.push_back(Round{0, first_file[G], 0, 1, 0});
        for (uint64_t b : row_bytes) rounds.back().bytes += b;
        return rounds;
    }
    uint32_t max_rows = kRoundMaxRows;
    if (const char* e = getenv("GRMKM_ROUND_ROWS")) max_rows = (uint32_t)std::min(16, std::max(1, atoi(e)));
    uint32_t r = 0;
    while (r < G) {
        Round rd{first_file[r], first_file[r + 1], r, 1, row_bytes[r]};
        while (rd.n_rows < max_rows && r + rd.n_rows < G && ((r + rd.n_rows) & 63u) != 0) {
            const uint32_t nr = rd.n_rows + 1;
            // (further rows join only while the round still needs no key sub-ranges: every sub-range bit doubles the
            // aggregate's passes over the round's records, and rows share nothing that would pay for it -- the distinct
            // k-mers of read sets are mostly sequencing errors, unique to their genome)
            const uint64_t cap_keys = (uint64_t)table_slots(c, (nr + 1) & ~1u) * 6 / 10 << kUnitMaxBucketBits;
            const uint64_t nb = rd.bytes + row_bytes[r + rd.n_rows];
            if (nb / 10 > cap_keys) break;
            rd.n_rows = nr; rd.bytes = nb; rd.f1 = first_file[r + nr];
        }
        rounds.push_back(rd);
        r += rd.n_rows;
    }
    return rounds;
}

// Bucket count: the distinct k-mers of a bucket must fit its shared-memory table at a load of about 0.6 by the
// estimate (a bucket that turns out too full is split into key sub-ranges by the kernel, so the estimate only costs
// time, never correctness).  Fewer buckets = longer runs per scatter tile = fewer store requests.  Past 2^11 buckets
// every further bit doubles the aggregate's passes over the records (key sub-ranges), so a table that the estimate
// fills to 0.7 is still the better deal.
uint32_t bits_for(uint64_t u_est, uint32_t slots) {
    const uint64_t per = std::max<uint64_t>(1, (uint64_t)slots * 60 / 100);
    uint32_t bits = std::min(kUnitMaxBucketBits + kMaxSubBits, std::max(6u, ceil_log2((u_est + per - 1) / per)));
    if (bits > kUnitMaxBucketBits) {
        const uint64_t per7 = std::max<uint64_t>(1, (uint64_t)slots * 70 / 100);
        if (ceil_log2((u_est + per7 - 1) / per7) <= kUnitMaxBucketBits) bits = kUnitMaxBucketBits;
    }
    return bits;
}

struct InputTable {
    uint32_t G = 0;
    std::vector<uint32_t> first_file;      // [G + 1] (inputs sorted by row)
    std::vector<uint64_t> row_bytes;       // [G]
    uint64_t max_row = 0, in_bytes = 0;
};

// sorts the inputs by genome row (stable: the files of a row keep their order) and tabulates them
InputTable tabulate_inputs(grmkm_ctx* c) {
    InputTable t;
    uint32_t maxrow = 0;
    for (const Input& in : c->inputs) maxrow = std::max(maxrow, in.row + 1);
    t.G = std::max(maxrow, c->n_genomes_decl);
    if (!(c->cfg.flags & GRMKM_FLAG_COUNTS) && (abundance_build(c) || t.G > kBlockRows))
        std::stable_sort(c->inputs.begin(), c->inputs.end(), [](const Input& a, const Input& b) { return a.row < b.row; });
    for (Input& in : c->inputs) if (!in.owned.empty()) in.host = in.owned.data();
    t.first_file.assign(t.G + 1, 0);
    t.row_bytes.assign(std::max(t.G, 1u), 0);
    for (const Input& in : c->inputs) { t.first_file[in.row + 1]++; t.row_bytes[in.row] += in.len; t.in_bytes += in.len; }
    for (uint32_t g = 0; g < t.G; ++g) t.first_file[g + 1] += t.first_file[g];
    for (uint64_t b : t.row_bytes) t.max_row = std::max(t.max_row, b);
    return t;
}

// the automatic bucket count of the inputs added so far (cfg.bucket_bits = 0); all ranks of a multi-GPU build agree on
// the maximum of theirs before they build (grmkm_plan_bucket_bits / grmkm_set_bucket_bits)
uint32_t auto_bucket_bits(grmkm_ctx* c, const InputTable& t) {
    if (!abundance_build(c)) {
        // the pan-genome of the context is estimated from the largest genome (1.9 x its text)
        const uint64_t u_est = t.max_row + t.max_row * 9 / 10 + 1024;
        return bits_for(u_est, table_slots(c, 2 * ((t.G + 63) / 64)));
    }
    uint64_t rb = 0; uint32_t rr = 1;
    for (const Round& rd : plan_rounds(c, t.G, t.first_file, t.row_bytes)) { rb = std::max(rb, rd.bytes); rr = std::max(rr, rd.n_rows); }
    return bits_for(rb / 12 + 1024, table_slots(c, (rr + 1) & ~1u));       // one distinct k-mer per 12 bytes of read text (measured: 12.4)
}

// ------------------------------------------------------------------------------------------------
// one pipeline pass over inputs [f0, f1): parse -> pack -> unit bounds -> unit scatter -> dedupe -> expand -> aggregate
// ------------------------------------------------------------------------------------------------
enum AggKind { AGG_FINAL = 4, AGG_PARTIAL = 5, AGG_ROUND = 6, AGG_COUNTS = 7 };

int check_ctx(const grmkm_ctx* c) { return c ? GRMKM_OK : GRMKM_E_INVALID; }

struct Geo {
    uint32_t G = 0, W = 0;                   // genomes / matrix word rows of the whole build
    uint32_t bucket_bits = 0, sub_bits = 0;  // hash buckets of the expansion, key sub-ranges of the aggregate
    uint32_t B = 0, VB = 0;
};

struct QueryJob;

struct Job {
    uint32_t f0 = 0, f1 = 0;        // inputs
    uint32_t row0 = 0, n_rows = 0;  // genome rows of the job (FileDesc.row = input row - row0)
    AggKind agg = AGG_FINAL;
    uint64_t max_row_bytes = 0;     // text of the job's largest genome row
    // AGG_ROUND: where the round's records go
    ulonglong2* round_out = nullptr;
    uint64_t round_cap = 0;
    // a query job (grmkm_query): every batch's packed stream goes through k_query_scan instead of the unit path, and
    // the job ends after the last batch
    const QueryJob* query = nullptr;
};

struct QueryJob {
    QueryScanParams sp;             // table, plane / counters, totals (the batch fields are filled per batch)
    bool smem = false, count = false;
    uint32_t ctas_per_sm = 1;
    size_t smem_bytes = 0;
};

int launch_query_scan(grmkm_ctx* c, const QueryJob& q, const FileDesc* d_files, uint32_t n_files, uint64_t n_groups_max) {
    QueryScanParams sp = q.sp;
    sp.codes = (const unsigned long long*)c->codes.p; sp.valid = (const uint32_t*)c->valid.p;
    sp.scalars = (const uint64_t*)c->scalars.p; sp.fss = (const uint64_t*)c->fss.p; sp.files = d_files; sp.n_files = n_files;
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((n_groups_max + kQsThreads - 1) / kQsThreads,
                                                                               (uint64_t)c->sm_count * q.ctas_per_sm));
    void (*kern)(QueryScanParams) = q.smem ? (q.count ? k_query_scan<true, true> : k_query_scan<true, false>)
                                           : (q.count ? k_query_scan<false, true> : k_query_scan<false, false>);
    kern<<<grid, kQsThreads, q.smem_bytes, c->stream>>>(sp);
    CU_TRY(c, cudaGetLastError());
    return GRMKM_OK;
}

struct JobOut {
    uint64_t sc[S_COUNT] = {0};
    uint64_t ucap = 0;
    uint64_t h2d = 0;
    uint32_t launches = 0, MB = 0;
    bool ordered = false;
    bool round_full = false;        // AGG_ROUND: the output did not fit round_cap (nothing else is wrong)
    std::vector<uint64_t> h_off;    // AGG_PARTIAL: offsets of the (virtual) bucket chunks
};

void add_stage_times(grmkm_ctx* c) {
    if (!c->ev_ok) return;
    float* t[] = {&c->times.h2d, &c->times.parse, &c->times.pack, &c->times.count, &c->times.bounds, &c->times.scatter,
                  &c->times.abundance, &c->times.dedupe, &c->times.expand, &c->times.aggregate, &c->times.sort};
    for (int i = 1; i < T_N; ++i) {
        float v = 0.f;
        const cudaError_t te = cudaEventElapsedTime(&v, c->ev[i - 1], c->ev[i]);
        if (te != cudaSuccess) {
            cudaGetLastError();
            if (getenv("GRMKM_DEBUG")) fprintf(stderr, "grmkm: stage event %d: %s\n", i, cudaGetErrorString(te));
            v = 0.f;
        }
        *t[i - 1] += v;
    }
    float tot = 0.f;
    if (cudaEventElapsedTime(&tot, c->ev[T_START], c->ev[T_SORT]) == cudaSuccess) c->times.total += tot; else cudaGetLastError();
}

// The column aggregate over bucketed wide records (final presence columns, partial columns, an abundance round or the
// pooled count table), with its retry when the output guess was too small.  Leaves the scalars in out.sc.
struct AggIn {
    const unsigned long long* records; const unsigned long long* begin; const unsigned long long* end;
    uint32_t wide_words, wide_stride, row_bits;     // record geometry
    uint32_t cells, n_words;                        // table cells per slot, words per output column
    AggKind agg;
    uint32_t round_rows = 0, round_row0 = 0, out_wbits = 0, out_word = 0;
    ulonglong2* round_out = nullptr;
    uint64_t ucap_guess = 0;
};

int run_aggregate(grmkm_ctx* c, const Geo& geo, const AggIn& in, JobOut& out, bool& retry_outer,
                  const std::function<int(const uint64_t*)>& check_upstream) {
    cudaStream_t st = c->stream;
    uint64_t* d_scalars = (uint64_t*)c->scalars.p;
    const uint32_t slots = table_slots(c, in.cells);
    if (slots < 256) return fail(c, GRMKM_E_UNSUPPORTED, "too many genomes for the shared-memory column table");
    const size_t smem = table_smem(slots, in.cells);
    const uint32_t VB = geo.VB;
    const uint32_t vgrid = std::min<uint32_t>(VB, (uint32_t)c->sm_count * kAggCtasPerSm);
    const bool final_like = in.agg == AGG_FINAL || in.agg == AGG_COUNTS;
    const bool ordered = final_like && !getenv("GRMKM_UNORDERED");
    out.ordered = ordered;
    // (an abundance round writes behind the earlier rounds' records: its capacity is what is left, possibly nothing)
    uint64_t ucap = std::min<uint64_t>(in.agg == AGG_ROUND ? in.ucap_guess : std::max<uint64_t>(in.ucap_guess, 1), 0xFFFFFFFFULL);
    ENSURE(c, c->bbase, (size_t)VB * 8);
    ENSURE(c, c->bcounts, (size_t)VB * 8);
    if (ordered) ENSURE(c, c->apub, (size_t)(VB + 1) * 8);
    retry_outer = false;
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (in.agg == AGG_ROUND) {
            // the records go straight behind the earlier rounds' (the caller grows that buffer when a round does not fit)
        } else if (ordered) {
            // the columns land at their final place: k-mers in the result array, word row w at matrix + w * ucap (the
            // result's row pitch is the capacity: no pass over the rows once U is known)
            ENSURE(c, c->kmers, ucap * 8);
            ENSURE(c, c->matrix, (size_t)ucap * in.n_words * 8);
            CU_TRY(c, cudaMemsetAsync(c->apub.p, 0, (size_t)(VB + 1) * 8, st));
        } else {
            ENSURE(c, c->ukeys, ucap * 8);
            ENSURE(c, c->uwords, (size_t)ucap * in.n_words * 8);
        }
        AggParams2 ap{};
        ap.records = in.records; ap.begin = in.begin; ap.end = in.end; ap.bucket_bits = geo.bucket_bits;
        ap.row_bits = in.row_bits; ap.n_words = in.n_words; ap.slots = slots;
        ap.keep_singletons = c->cfg.keep_singletons; ap.sub_bits = geo.sub_bits;
        ap.wide_words = in.wide_words; ap.wide_stride = in.wide_stride; ap.table_u32 = in.cells;
        ap.out_keys = (unsigned long long*)c->ukeys.p; ap.out_words = (unsigned long long*)c->uwords.p;
        ap.cap = ucap; ap.scalars = (unsigned long long*)d_scalars;
        ap.bucket_base = (unsigned long long*)c->bbase.p; ap.bucket_count = (unsigned long long*)c->bcounts.p;
        ap.b_begin = 0; ap.b_end = geo.B;
        ap.min_abundance = c->cfg.min_abundance; ap.round_rows = in.round_rows; ap.round_row0 = in.round_row0;
        ap.out_wbits = in.out_wbits; ap.out_word = in.out_word; ap.out_wide = in.round_out;
        if (ordered) {
            ap.ordered = 1;
            ap.out_keys = (unsigned long long*)c->kmers.p; ap.out_words = (unsigned long long*)c->matrix.p;
            ap.pub = (unsigned long long*)c->apub.p; ap.ticket = (unsigned int*)((unsigned long long*)c->apub.p + VB);
        }
        void (*kern)(AggParams2) = in.agg == AGG_FINAL ? k_aggregate_cols<4> : in.agg == AGG_PARTIAL ? k_aggregate_cols<5>
                                   : in.agg == AGG_ROUND ? k_aggregate_cols<6> : k_aggregate_cols<7>;
        CU_TRY(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<vgrid, kAggThreads, smem, st>>>(ap);
        out.launches++;
        CU_TRY(c, cudaGetLastError());
        if (ordered && c->ev_ok) cudaEventRecord(c->ev[T_AGG], st);
        CU_TRY(c, cudaMemcpyAsync(out.sc, d_scalars, sizeof out.sc, cudaMemcpyDeviceToHost, st));
        CU_TRY(c, cudaStreamSynchronize(st));
        const int up = check_upstream(out.sc);          // 1: an upstream guess was too small, the caller repeats the round
        if (up < 0) return up;
        if (up > 0) { retry_outer = true; break; }
        if (out.sc[S_U_NEEDED] <= ucap) break;
        if (in.agg == AGG_ROUND) { out.round_full = true; break; }
        if (attempt == 1 || out.sc[S_U_NEEDED] > 0xFFFFFFFFULL)
            return fail(c, GRMKM_E_UNSUPPORTED, "more than 2^32 columns in one context");
        ucap = out.sc[S_U_NEEDED];
        const uint64_t zero3[3] = {0, 0, 0};
        CU_TRY(c, cudaMemcpyAsync(d_scalars + S_U_NEEDED, zero3, 3 * 8, cudaMemcpyHostToDevice, st));     // + S_N_DISTINCT, S_N_SPLITS
        CU_TRY(c, cudaStreamSynchronize(st));           // zero3 lives on this stack frame
    }
    out.ucap = ucap;
    return GRMKM_OK;
}

int run_job(grmkm_ctx* c, const Geo& geo, const Job& job, JobOut& out) {
    cudaStream_t st = c->stream;
    const bool counting = job.agg == AGG_ROUND || job.agg == AGG_COUNTS;
    const uint32_t B = geo.B;

    // ---- batches.  Host inputs are staged batch by batch on a copy stream (two staging halves), so that the
    // H2D copy of batch i+1 overlaps parse / pack / scatter of batch i; the scatter appends to the bucket
    // regions, so batches need no merge.  Device-resident inputs (and the exact-offset fallback, which needs
    // a count over everything first) run as one batch.
    struct Batch { uint32_t f0, f1; uint64_t bytes, staged, tiles, stream; };
    // stream entries reserved for a file: every byte yields at most one entry; files start on group boundaries
    auto stream_cap = [](uint64_t len) { return ((len + 31) & ~31ULL) + 32; };
    bool any_host = false;
    uint64_t max_stream = 0, in_bytes = 0;
    for (uint32_t f = job.f0; f < job.f1; ++f) {
        const Input& in = c->inputs[f];
        max_stream += stream_cap(in.len); in_bytes += in.len; any_host = any_host || !in.dev;
    }
    auto make_batches = [&](bool pipelined) {
        std::vector<Batch> v;
        const uint64_t target = pipelined ? c->batch_bytes : ~0ULL;
        Batch cur{job.f0, job.f0, 0, 0, 0, 0};
        for (uint32_t f = job.f0; f < job.f1; ++f) {
            const Input& in = c->inputs[f];
            if (cur.f1 > cur.f0 && cur.bytes + in.len > target) { v.push_back(cur); cur = Batch{f, f, 0, 0, 0, 0}; }
            cur.f1 = f + 1; cur.bytes += in.len; cur.stream += stream_cap(in.len);
            if (!in.dev) cur.staged += (in.len + 15) & ~15ULL;
            cur.tiles += std::max<uint64_t>(1, (in.len + kTileBytes - 1) / kTileBytes);
        }
        v.push_back(cur);
        return v;
    };

    ENSURE(c, c->scalars, S_COUNT * 8);
    ENSURE(c, c->hist, (size_t)B * 8 * kCursorStride);
    ENSURE(c, c->offsets, (size_t)(B + 1) * 8);
    uint64_t* d_scalars = (uint64_t*)c->scalars.p;
    const FileDesc* d_files = nullptr;

    const bool query = job.query != nullptr;
    if (c->ev_ok && !query) cudaEventRecord(c->ev[T_START], st);
    CU_TRY(c, cudaMemsetAsync(c->scalars.p, 0, S_COUNT * 8, st));

    // parse + pack of one batch: leaves codes / valid / fss / S_STREAM_LEN of the batch
    auto front = [&](const Batch& bt, const uint8_t* staged_base, bool timed) -> int {
        const uint32_t F = bt.f1 - bt.f0;
        const uint64_t n_tiles = bt.tiles;
        const uint64_t n_groups_max = bt.stream / 32 + 2;
        if (n_tiles > 0x7fffffffULL) return fail(c, GRMKM_E_UNSUPPORTED, "input too large for one build (tile count)");
        ENSURE(c, c->files, F * sizeof(FileDesc));
        ENSURE(c, c->hdr0, F * 8);
        ENSURE(c, c->fss, (F + 1) * 8);
        ENSURE(c, c->tile_file, n_tiles * sizeof(TileTicket));
        ENSURE(c, c->tile_pub, (3 * n_tiles + 1) * 8);    // published tile summaries / states (look-back) + the ticket counter
        ENSURE(c, c->codes, n_groups_max * 8);
        ENSURE(c, c->valid, n_groups_max * 4);
        ENSURE(c, c->tile_order, n_tiles * 4);
        // the memsets go first: the device clears while the host builds this batch's tables -- unless the previous build
        // already cleared the buffers on the side stream (same buffers, at least this much of them)
        bool cleared = false;
        if (c->pre_pending) {
            CU_TRY(c, cudaStreamWaitEvent(st, c->ev_cleared, 0));
            cleared = c->pre_codes == c->codes.p && c->pre_valid == c->valid.p && c->pre_pub == c->tile_pub.p &&
                      c->pre_groups >= n_groups_max && c->pre_pub_bytes >= (3 * n_tiles + 1) * 8;
            c->pre_pending = false;
        }
        if (!cleared) {
            CU_TRY(c, cudaMemsetAsync(c->codes.p, 0, n_groups_max * 8, st));
            CU_TRY(c, cudaMemsetAsync(c->valid.p, 0, n_groups_max * 4, st));
            CU_TRY(c, cudaMemsetAsync(c->tile_pub.p, 0, (3 * n_tiles + 1) * 8, st));
        }
        c->pass_groups = std::max<uint64_t>(c->pass_groups, n_groups_max);
        c->pass_pub_bytes = std::max<uint64_t>(c->pass_pub_bytes, (3 * n_tiles + 1) * 8);
        // host tables in page-locked memory (asynchronous copies without a staging hop); they stay untouched until the
        // build's final synchronize
        const size_t tab_bytes = (F * sizeof(FileDesc) + (F + 1) * 8 + (size_t)n_tiles * 4 + 63) & ~size_t(63);
        if (c->h_tab_used + tab_bytes > c->h_tab_cap) return fail(c, GRMKM_E_NOMEM, "host table arena too small");
        uint8_t* tab = (uint8_t*)c->h_tab + c->h_tab_used;
        c->h_tab_used += tab_bytes;
        FileDesc* fds = (FileDesc*)tab;
        uint64_t* fss = (uint64_t*)(tab + F * sizeof(FileDesc));      // where every file's entries start in the stream
        uint32_t* order = (uint32_t*)(fss + F + 1);                   // ticket -> tile: round-robin over the files
        uint64_t tiles = 0, soff = 0, spos = 0;
        std::vector<std::pair<uint64_t, uint32_t>> by_tiles(F);       // (tile count, file), most tiles first
        for (uint32_t i = 0; i < F; ++i) {
            const Input& in = c->inputs[bt.f0 + i];
            fds[i].len = in.len; fds[i].row = in.row - job.row0; fds[i].kind = in.kind; fds[i].tile_begin = tiles;
            const uint64_t nt = std::max<uint64_t>(1, (in.len + kTileBytes - 1) / kTileBytes);
            by_tiles[i] = {nt, i};
            tiles += nt;
            fss[i] = spos; spos += stream_cap(in.len);
            if (in.dev) fds[i].ptr = in.dev;
            else { fds[i].ptr = staged_base + soff; soff += (in.len + 15) & ~15ULL; }
        }
        fss[F] = spos;
        std::sort(by_tiles.begin(), by_tiles.end(), [](const std::pair<uint64_t, uint32_t>& a, const std::pair<uint64_t, uint32_t>& b) {
            return a.first != b.first ? a.first > b.first : a.second < b.second; });
        {
            size_t o = 0, live = F;                                    // files that still have a tile number `l`
            for (uint64_t l = 0; o < n_tiles; ++l) {
                while (live > 0 && by_tiles[live - 1].first <= l) --live;
                for (size_t q = 0; q < live; ++q) order[o++] = (uint32_t)(fds[by_tiles[q].second].tile_begin + l);
            }
        }
        d_files = (const FileDesc*)c->files.p;
        CU_TRY(c, cudaMemcpyAsync(c->files.p, fds, F * sizeof(FileDesc), cudaMemcpyHostToDevice, st));
        CU_TRY(c, cudaMemcpyAsync(c->fss.p, fss, (F + 1) * 8, cudaMemcpyHostToDevice, st));
        CU_TRY(c, cudaMemcpyAsync(c->tile_order.p, order, n_tiles * 4, cudaMemcpyHostToDevice, st));
        if (timed && c->ev_ok) cudaEventRecord(c->ev[T_H2D], st);
        k_first_header<<<(F * 32 + 255) / 256, 256, 0, st>>>(d_files, F, (uint64_t*)c->hdr0.p);
        k_tile_tickets<<<(uint32_t)((n_tiles + 255) / 256), 256, 0, st>>>(d_files, F, (const uint64_t*)c->hdr0.p, (const uint64_t*)c->fss.p,
                                                                           (const uint32_t*)c->tile_order.p, n_tiles, (TileTicket*)c->tile_file.p);
        out.launches += 2;
        CU_TRY(c, cudaGetLastError());
        if (timed && c->ev_ok) cudaEventRecord(c->ev[T_PARSE], st);
        // single pass: summaries are published and resolved by look-back inside k_pack (grmkm_kernels.cuh)
        PackParams pp{};
        pp.files = d_files; pp.hdr0 = (const uint64_t*)c->hdr0.p; pp.n_tiles = n_tiles; pp.n_files = F;
        pp.tickets = (const TileTicket*)c->tile_file.p; pp.ticket = (uint32_t*)((unsigned long long*)c->tile_pub.p + 3 * n_tiles);
        pp.pub_a0 = (unsigned long long*)c->tile_pub.p; pp.pub_a1 = pp.pub_a0 + n_tiles; pp.pub_ps = pp.pub_a0 + 2 * n_tiles;
        pp.stream_len = bt.stream;
        pp.codes = (unsigned long long*)c->codes.p; pp.valid = (uint32_t*)c->valid.p; pp.scalars = d_scalars;
        const auto pack = c->cfg.input_kind == GRMKM_FASTA ? k_pack<0> : k_pack<1>;
        pack<<<(uint32_t)n_tiles, kParseThreads, 0, st>>>(pp);
        out.launches++;
        CU_TRY(c, cudaGetLastError());
        if (timed && c->ev_ok) cudaEventRecord(c->ev[T_PACK], st);
        return GRMKM_OK;
    };

    // ---- unit (super-k-mer) geometry (grmkm_units.cuh).  Presence: a dedupe entry / wide record holds WB presence
    // words of one genome group.  Abundance: the "group" is the job-local genome row and the word a count.
    const UnitGeom ug = unit_geom(c->cfg.k);
    const uint32_t WB = counting ? 1u : unit_words_per_entry(geo.W);
    const uint32_t n_groups_w = counting ? std::max(1u, job.n_rows) : (geo.W + WB - 1) / WB;
    const uint32_t wbits = std::max(1u, ceil_log2(n_groups_w));
    if (!query && wbits > geo.bucket_bits) return fail(c, GRMKM_E_UNSUPPORTED, "more genome groups than hash buckets");
    const uint32_t ES = 2 + WB, RS = unit_record_stride(WB);
    uint32_t MB = (uint32_t)c->sm_count;
    if (!query) {
        // distinct (unit, genome group) entries of a bucket should fit the dedupe table about once
        const uint64_t entries = counting ? in_bytes / (ug.w + 1) / 2 + 1
                                          : (job.max_row_bytes * 19 / 10) * 2 / (ug.w + 1) * 13 / 10 * n_groups_w;
        const uint64_t per_wave = (uint64_t)unit_dedupe_slots(WB) * 6 / 10 * c->sm_count;
        const uint64_t waves = std::max<uint64_t>(1, (entries + per_wave - 1) / per_wave);
        MB = (uint32_t)std::min<uint64_t>(kUsMaxBuckets, waves * c->sm_count);
        if (const char* ub = getenv("GRMKM_UNIT_BUCKETS")) MB = (uint32_t)std::min(kUsMaxBuckets, std::max(1, atoi(ub)));
        ENSURE(c, c->ucur, (size_t)MB * 8);
        ENSURE(c, c->ubeg, (size_t)(MB + 1) * 8);
    }
    out.MB = MB;
    const bool try_regions = !getenv("GRMKM_EXACT_OFFSETS");
    uint64_t* sc = out.sc;
    // codes / valid / tile words are dead once the last batch has been scattered (or scanned): clear them for the next
    // build or query (or the next pass) on the side stream, under whatever the stream runs next
    auto preclear = [&]() -> int {
        if (!c->pass_groups) return GRMKM_OK;
        if (!c->aux_stream) {
            CU_TRY(c, cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking));
            CU_TRY(c, cudaEventCreateWithFlags(&c->ev_scattered, cudaEventDisableTiming));
            CU_TRY(c, cudaEventCreateWithFlags(&c->ev_cleared, cudaEventDisableTiming));
        }
        CU_TRY(c, cudaEventRecord(c->ev_scattered, st));
        CU_TRY(c, cudaStreamWaitEvent(c->aux_stream, c->ev_scattered, 0));
        CU_TRY(c, cudaMemsetAsync(c->codes.p, 0, c->pass_groups * 8, c->aux_stream));
        CU_TRY(c, cudaMemsetAsync(c->valid.p, 0, c->pass_groups * 4, c->aux_stream));
        CU_TRY(c, cudaMemsetAsync(c->tile_pub.p, 0, c->pass_pub_bytes, c->aux_stream));
        CU_TRY(c, cudaEventRecord(c->ev_cleared, c->aux_stream));
        c->pre_pending = true;
        c->pre_codes = c->codes.p; c->pre_valid = c->valid.p; c->pre_pub = c->tile_pub.p;
        c->pre_groups = c->pass_groups; c->pre_pub_bytes = c->pass_pub_bytes;
        return GRMKM_OK;
    };
    for (int pass = try_regions ? 0 : 1; pass < 2; ++pass) {
        // Pass 0 scatters into over-provisioned bucket regions without a count pass; if a region overflows (heavily
        // skewed unit spectrum) pass 1 redoes the scatter with exact offsets from a count pass.
        const bool regions = (pass == 0);
        c->pass_groups = 0; c->pass_pub_bytes = 0;
        const std::vector<Batch> batches = make_batches(regions && any_host);
        const bool pipelined = batches.size() > 1;
        {   // host table arena for all batches of this pass (nothing of an earlier pass / build is in flight: both end synchronised)
            size_t need = 0;
            for (const Batch& bt : batches)
                need += (((size_t)(bt.f1 - bt.f0) * sizeof(FileDesc) + (bt.f1 - bt.f0 + 1) * 8 + (size_t)bt.tiles * 4 + 63) & ~size_t(63));
            if (need > c->h_tab_cap) {
                CU_TRY(c, cudaStreamSynchronize(st));
                if (c->h_tab) cudaFreeHost(c->h_tab);
                c->h_tab = nullptr; c->h_tab_cap = 0;
                CU_TRY(c, cudaHostAlloc(&c->h_tab, need + need / 4, cudaHostAllocDefault));
                c->h_tab_cap = need + need / 4;
            }
            c->h_tab_used = 0;
        }
        uint64_t cap = 0;
        if (query) {
            // (no unit regions: the scan writes the plane)
        } else if (regions) {
            const double est_units = (double)max_stream * 2.0 / (ug.w + 1) * 1.15;
            cap = (uint64_t)(est_units / MB * 1.25) + 4096;
            cap = (cap + 15) & ~15ULL;
            ENSURE(c, c->units, ((uint64_t)MB * cap + kUsStage) * 16);
        } else {
            ENSURE(c, c->units, (max_stream + kUsStage) * 16);
        }
        uint64_t half_bytes = 0;
        for (const Batch& bt : batches) half_bytes = std::max(half_bytes, bt.staged);
        ENSURE(c, c->in, half_bytes * (pipelined ? 2 : 1));
        if (pipelined && !c->copy_stream) {
            CU_TRY(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
            for (int i = 0; i < 2; ++i) {
                CU_TRY(c, cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
                CU_TRY(c, cudaEventCreateWithFlags(&c->ev_free[i], cudaEventDisableTiming));
            }
        }
        CU_TRY(c, cudaMemsetAsync(d_scalars, 0, S_COUNT * 8, st));
        if (regions && !query) {
            k_init_regions<<<(MB + 1 + 255) / 256, 256, 0, st>>>((unsigned long long*)c->ubeg.p, (unsigned long long*)c->ucur.p, MB, cap);
            out.launches++;
        }
        if (pipelined && c->ev_ok && !query)
            for (int e : {T_H2D, T_PARSE, T_PACK, T_COUNT, T_BOUNDS}) cudaEventRecord(c->ev[e], st);   // stages interleave: only "scatter" is timed
        out.h2d = 0;
        NvtxRange nv_front("grmkm front: stage / pack / unit bounds / unit scatter");
        std::unique_lock<std::mutex> gate;
        cudaEvent_t* gate_ev = nullptr;
        if (any_host && c->device >= 0 && c->device < 64) {
            gate = std::unique_lock<std::mutex>(g_h2d.mu);
            gate_ev = &g_h2d.done[c->device];
            if (!*gate_ev) CU_TRY(c, cudaEventCreateWithFlags(gate_ev, cudaEventDisableTiming));
            else CU_TRY(c, cudaStreamWaitEvent(pipelined ? c->copy_stream : st, *gate_ev, 0));
        }
        for (size_t bi = 0; bi < batches.size(); ++bi) {
            const Batch& bt = batches[bi];
            uint8_t* half = (uint8_t*)c->in.p + (pipelined ? (bi & 1) * half_bytes : 0);
            cudaStream_t cs = pipelined ? c->copy_stream : st;
            if (pipelined && bi >= 2) CU_TRY(c, cudaStreamWaitEvent(cs, c->ev_free[bi & 1], 0));
            // Host buffers that follow one another in memory the way they are staged (each padded to 16 bytes: the arena of
            // create._read_inputs, bench.py) travel as ONE copy per batch.  A train of 5 MB copies loses the link to a large
            // copy in the other direction (another context's result on its way out: profiles/r02_duplex_pattern.txt).
            uint64_t soff = 0, run_dst = 0, run_len = 0;
            const uint8_t* run_src = nullptr;
            auto flush_run = [&]() -> int {
                if (run_len) CU_TRY(c, cudaMemcpyAsync(half + run_dst, run_src, run_len, cudaMemcpyHostToDevice, cs));
                run_len = 0; run_src = nullptr;
                return GRMKM_OK;
            };
            for (uint32_t f = bt.f0; f < bt.f1; ++f) {
                const Input& in = c->inputs[f];
                if (in.dev) continue;
                const uint64_t padded = (in.len + 15) & ~15ULL;
                if (in.len) {
                    if (run_len && in.host == run_src + (soff - run_dst)) run_len = (soff - run_dst) + in.len;      // adjacent: extend the run
                    else { int fr = flush_run(); if (fr) return fr; run_src = in.host; run_dst = soff; run_len = in.len; }
                    out.h2d += in.len;
                }
                soff += padded;
            }
            { int fr = flush_run(); if (fr) return fr; }
            if (pipelined) {
                CU_TRY(c, cudaEventRecord(c->ev_copied[bi & 1], cs));
                CU_TRY(c, cudaStreamWaitEvent(st, c->ev_copied[bi & 1], 0));
            }
            int fr = front(bt, half, !pipelined && !query);
            if (fr) return fr;
            if (pipelined) CU_TRY(c, cudaEventRecord(c->ev_free[bi & 1], st));     // the staged text has been consumed
            if (query) {
                fr = launch_query_scan(c, *job.query, d_files, bt.f1 - bt.f0, bt.stream / 32 + 2);
                if (fr) return fr;
                out.launches++;
                continue;
            }

            const uint32_t F = bt.f1 - bt.f0;
            const uint64_t n_groups_max = bt.stream / 32 + 2;
            ENSURE(c, c->masks, n_groups_max * 8);
            const uint64_t n_utiles = (n_groups_max + kUsTileGroups - 1) / kUsTileGroups;
            ENSURE(c, c->stile_file, n_utiles * 4);
            if (!pipelined && c->ev_ok) cudaEventRecord(c->ev[T_COUNT], st);
            // two groups per thread and step, grid-stride (the next pair's words are fetched ahead): 8 CTAs' worth per SM
            const uint32_t bgrid = (uint32_t)std::min<uint64_t>((n_groups_max + 511) / 512, (uint64_t)c->sm_count * 8);
#define GRMKM_BOUNDS(WW)                                                                                        \
    k_unit_bounds<WW><<<bgrid, 256, 0, st>>>((const unsigned long long*)c->codes.p, (const uint32_t*)c->valid.p, d_scalars, \
                                             ug.k, ug.m, (uint2*)c->masks.p)
            switch (ug.w) {
                case 21: GRMKM_BOUNDS(21); break;
                case 13: GRMKM_BOUNDS(13); break;
                case 7: GRMKM_BOUNDS(7); break;
                case 4: GRMKM_BOUNDS(4); break;
                case 2: GRMKM_BOUNDS(2); break;
                default: GRMKM_BOUNDS(1); break;
            }
#undef GRMKM_BOUNDS
            k_stream_tile_files<<<(uint32_t)((n_utiles + 255) / 256), 256, 0, st>>>(
                d_scalars, (const uint64_t*)c->fss.p, F, (uint32_t*)c->stile_file.p, n_utiles, (uint64_t)kUsTileGroups * 32);
            out.launches += 2;
            CU_TRY(c, cudaGetLastError());
            if (!pipelined && c->ev_ok) cudaEventRecord(c->ev[T_BOUNDS], st);
            UnitScatterParams up{};
            up.codes = (const unsigned long long*)c->codes.p; up.masks = (const uint2*)c->masks.p; up.scalars = d_scalars;
            up.file_stream_start = (const uint64_t*)c->fss.p; up.files = d_files; up.tile_file = (const uint32_t*)c->stile_file.p;
            up.n_files = F; up.k = ug.k; up.lmax = ug.lmax; up.n_buckets = MB;
            up.cursors = (unsigned long long*)c->ucur.p; up.units = (uint4*)c->units.p; up.cap = cap;
            up.dump = (uint64_t)MB * cap; up.overflow = (unsigned long long*)(d_scalars + S_OVERFLOW);
            up.n_windows = (unsigned long long*)(d_scalars + S_N_WINDOWS);
            const size_t usm = unit_scatter_smem(MB);
            const uint32_t ugrid = (uint32_t)std::min<uint64_t>(n_utiles, (uint64_t)c->sm_count);
            if (!regions) {
                CU_TRY(c, cudaMemsetAsync(c->ucur.p, 0, (size_t)MB * 8, st));
                CU_TRY(c, cudaFuncSetAttribute(k_units_scatter<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)usm));
                k_units_scatter<true><<<ugrid, kUsThreads, usm, st>>>(up);
                k_bucket_offsets<<<1, 1024, 0, st>>>((unsigned long long*)c->ucur.p, (unsigned long long*)c->ubeg.p, MB,
                                                     d_scalars, S_N_UNITS, 1);
                out.launches += 2;
            }
            CU_TRY(c, cudaFuncSetAttribute(k_units_scatter<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)usm));
            k_units_scatter<false><<<ugrid, kUsThreads, usm, st>>>(up);
            out.launches++;
            CU_TRY(c, cudaGetLastError());
        }
        if (gate_ev) {
            CU_TRY(c, cudaEventRecord(*gate_ev, pipelined ? c->copy_stream : st));      // behind this build's last copy
            gate.unlock();
        }
        if (query) return preclear();
        // bucket b = units[begin[b], end[b]): end = the cursors (clamped to the region)
        k_finish_unit_regions<<<1, 1024, 0, st>>>((const unsigned long long*)c->ubeg.p, (unsigned long long*)c->ucur.p, MB,
                                                  cap, (unsigned long long*)d_scalars, S_N_UNITS);
        out.launches++;
        CU_TRY(c, cudaGetLastError());
        if (c->ev_ok) cudaEventRecord(c->ev[T_SCATTER], st);
        // (under the dedupe / expand / aggregate kernels, which leave most of the HBM bandwidth unused)
        { const int pr = preclear(); if (pr) return pr; }

        nv_front.end();
        NvtxRange nv_back("grmkm back: dedupe / expand / aggregate");
        // Dedupe -> expand -> aggregate run back to back without a host round trip.  The dedupe's entry list and the
        // expansion's bucket regions are sized from estimates; the one synchronisation after the aggregate reads what
        // was really needed, and a guess that was too small repeats the round (entry list: larger; regions: exact
        // offsets from a count pass).
        const unsigned long long* agg_begin = (const unsigned long long*)c->offsets.p;
        const unsigned long long* agg_end = (const unsigned long long*)c->hist.p;
        uint64_t wcap = std::min<uint64_t>(max_stream, std::max<uint64_t>(1 << 16, max_stream / 16));
        bool wide_exact = !try_regions;
        if (getenv("GRMKM_WIDE_EXACT")) wide_exact = true;
        if (const char* e = getenv("GRMKM_WU_CAP")) wcap = std::max<uint64_t>(16, (uint64_t)atoll(e));     // tests: force the retry
        bool again = true, unit_overflow = false;
        for (int round = 0; again; ++round) {
            again = false;
            if (round > 6) return fail(c, GRMKM_E_UNSUPPORTED, "unit path does not converge");
            if (round > 0) {
                const uint64_t zero3[3] = {0, 0, 0};
                CU_TRY(c, cudaMemcpyAsync(d_scalars + S_U_NEEDED, zero3, 3 * 8, cudaMemcpyHostToDevice, st));      // + S_N_DISTINCT, S_N_SPLITS
                CU_TRY(c, cudaMemcpyAsync(d_scalars + S_WU_NEEDED, zero3, 3 * 8, cudaMemcpyHostToDevice, st));     // + S_N_WIDE, S_WIDE_OVERFLOW
                CU_TRY(c, cudaStreamSynchronize(st));          // zero3 lives on this stack frame
            }
            if (c->ev_ok) cudaEventRecord(c->ev[T_ABUND], st);
            const size_t dsm = unit_dedupe_smem(WB), xsm = staged_smem_bytes(B);
            void (*k_dedupe)(UnitDedupeParams) = counting ? k_units_dedupe<1, true>
                                                 : WB == 1 ? k_units_dedupe<1, false> : WB == 2 ? k_units_dedupe<2, false> : k_units_dedupe<4, false>;
            void (*k_xcount)(UnitExpandParams) = WB == 1 ? k_units_expand<true, 1> : WB == 2 ? k_units_expand<true, 2> : k_units_expand<true, 4>;
            void (*k_xscat)(UnitExpandParams) = WB == 1 ? k_units_expand<false, 1> : WB == 2 ? k_units_expand<false, 2> : k_units_expand<false, 4>;
            CU_TRY(c, cudaFuncSetAttribute(k_dedupe, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsm));
            CU_TRY(c, cudaFuncSetAttribute(k_xcount, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xsm));
            CU_TRY(c, cudaFuncSetAttribute(k_xscat, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xsm));
            // ---- dedupe: distinct (unit, group) entries
            ENSURE(c, c->wu, wcap * ES * 8);
            UnitDedupeParams dp{};
            dp.units = (const uint4*)c->units.p; dp.begin = (const unsigned long long*)c->ubeg.p;
            dp.end = (const unsigned long long*)c->ucur.p; dp.n_buckets = MB; dp.out = (unsigned long long*)c->wu.p;
            dp.cap = wcap; dp.needed = (unsigned long long*)(d_scalars + S_WU_NEEDED);
            k_dedupe<<<std::min<uint32_t>(MB, (uint32_t)c->sm_count), kUdThreads, dsm, st>>>(dp);
            out.launches++;
            CU_TRY(c, cudaGetLastError());
            if (c->ev_ok) cudaEventRecord(c->ev[T_DEDUPE], st);
            // ---- expand: every distinct entry -> wide records of its k-mers, by hash bucket
            UnitExpandParams xp{};
            xp.wu = (const unsigned long long*)c->wu.p; xp.n_ptr = (const unsigned long long*)(d_scalars + S_WU_NEEDED);
            xp.cap = wcap; xp.k = c->cfg.k; xp.bucket_bits = geo.bucket_bits; xp.wbits = wbits;
            xp.cursors = (unsigned long long*)c->hist.p; xp.records = nullptr;
            xp.overflow = (unsigned long long*)(d_scalars + S_WIDE_OVERFLOW);
            const uint32_t xgrid = (uint32_t)std::min<uint64_t>((wcap + kStThreads - 1) / kStThreads, (uint64_t)c->sm_count);
            if (!wide_exact) {
                // over-provisioned bucket regions, no count pass.  Presence: the distinct k-mers are estimated as 1.9 x the
                // largest genome plus 5 % of all input (what every further genome adds to a species' pan-genome), 1.3
                // records per distinct k-mer and genome group.  Abundance: every distinct (unit, genome) pair expands,
                // about a quarter of the text for reads, all of it for contigs.  1.4 x headroom per bucket; the previous
                // build (or round) of this context corrects the guess.
                uint64_t est;
                if (counting) est = c->cfg.input_kind == GRMKM_FASTQ ? in_bytes / 4 + 4096 : in_bytes + in_bytes / 8 + 4096;
                else est = std::min<uint64_t>(in_bytes, job.max_row_bytes * 19 / 10 + in_bytes / 20) * 13 / 10 * n_groups_w;
                est = std::max<uint64_t>(est, c->wide_hint);
                if (const char* wc = getenv("GRMKM_WIDE_EST")) est = (uint64_t)atoll(wc);
                // (rounded BEFORE the capacity test: tested unrounded, the size asked for was always a little more than the
                // size allocated, and cudaMemGetInfo -- a driver round trip that takes anything from 0.1 to 90 ms while the
                // GPU waits for the next launch -- ran in every build)
                uint64_t rcap = std::max<uint64_t>(64, ((uint64_t)((double)est / B * 1.4) + 1024) & ~15ULL);
                const uint64_t wide_need = ((uint64_t)B * rcap + kStTile) * RS * 8;
                if (wide_need > c->wide.cap) {
                    // the buffer has to grow: never beyond a quarter of what is free (a region that turns out too small
                    // only costs the count pass).  Not asked in the steady state -- cudaMemGetInfo is slow.
                    size_t free_b = 0, total_b = 0;
                    if (c->wide.cap && wide_need <= c->wide_capped_need) {
                        // a request this large was already cut down to what the context holds now: keep the buffer
                        rcap = std::min<uint64_t>(rcap, (c->wide.cap / (RS * 8) - kStTile) / B);
                    } else if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess) {
                        // (what it has already counts as the budget when that is more: no re-allocation every build)
                        const uint64_t have = std::max<uint64_t>(c->wide.cap, free_b / 4);
                        if (wide_need > have) c->wide_capped_need = wide_need;
                        rcap = std::min<uint64_t>(rcap, (have / (RS * 8) - kStTile) / B);
                    }
                }
                rcap = std::max<uint64_t>(64, rcap & ~15ULL);
                ENSURE(c, c->wide, ((uint64_t)B * rcap + kStTile) * RS * 8);
                k_init_regions<<<(B + 1 + 255) / 256, 256, 0, st>>>((unsigned long long*)c->offsets.p, (unsigned long long*)c->hist.p, B, rcap);
                xp.records = (unsigned long long*)c->wide.p; xp.region_cap = rcap; xp.dump = (uint64_t)B * rcap;
                k_xscat<<<xgrid, kStThreads, xsm, st>>>(xp);
                k_finish_regions<<<1, 1024, 0, st>>>((const unsigned long long*)c->offsets.p, (unsigned long long*)c->hist.p, B, rcap,
                                                     (unsigned long long*)d_scalars, S_N_WIDE);
                out.launches += 3;
                CU_TRY(c, cudaGetLastError());
                agg_begin = (const unsigned long long*)c->offsets.p;
                agg_end = (const unsigned long long*)c->hist.p;
            } else {
                // exact offsets: count pass, scan, one synchronisation to size the record array
                CU_TRY(c, cudaMemsetAsync(c->hist.p, 0, (size_t)B * 8, st));
                k_xcount<<<xgrid, kStThreads, xsm, st>>>(xp);
                k_bucket_offsets<<<1, 1024, 0, st>>>((unsigned long long*)c->hist.p, (unsigned long long*)c->offsets.p, B,
                                                     d_scalars, S_N_WIDE, kCursorStride);
                out.launches += 2;
                CU_TRY(c, cudaGetLastError());
                CU_TRY(c, cudaMemcpyAsync(sc, d_scalars, sizeof out.sc, cudaMemcpyDeviceToHost, st));
                CU_TRY(c, cudaStreamSynchronize(st));
                if (regions && sc[S_OVERFLOW]) { unit_overflow = true; break; }
                if (sc[S_WU_NEEDED] > wcap) {
                    // the entry count depends on the order the table fills in (bypass, flush points): leave headroom
                    wcap = sc[S_WU_NEEDED] + sc[S_WU_NEEDED] / 4 + 4096;
                    again = true;
                    continue;
                }
                ENSURE(c, c->wide, (sc[S_N_WIDE] + 1) * RS * 8);
                xp.records = (unsigned long long*)c->wide.p;
                k_xscat<<<xgrid, kStThreads, xsm, st>>>(xp);
                out.launches++;
                CU_TRY(c, cudaGetLastError());
                agg_begin = (const unsigned long long*)c->offsets.p;
                agg_end = agg_begin + 1;
            }
            if (c->ev_ok) cudaEventRecord(c->ev[T_EXPAND], st);

            // ---- aggregate.  Columns: three pan-genome estimates (1.9 x the largest genome each) + 1 % of all input, at
            // most a quarter of the windows (N / 4 alone asked for 163 GB of word rows at 1000 genomes); a guess that is
            // too small is retried with the exact number.
            AggIn ai{};
            ai.records = (const unsigned long long*)c->wide.p; ai.begin = agg_begin; ai.end = agg_end;
            ai.wide_words = WB; ai.wide_stride = RS; ai.row_bits = wbits; ai.agg = job.agg;
            if (job.agg == AGG_ROUND) {
                ai.cells = (job.n_rows + 1) & ~1u; ai.n_words = 1;
                ai.round_rows = job.n_rows; ai.round_row0 = job.row0;
                ai.out_wbits = std::max(1u, ceil_log2(geo.W)); ai.out_word = job.row0 >> 6;
                ai.round_out = job.round_out; ai.ucap_guess = job.round_cap;
            } else if (job.agg == AGG_COUNTS) {
                ai.cells = 2; ai.n_words = 1; ai.round_rows = 1; ai.round_row0 = 0;
                ai.ucap_guess = std::min<uint64_t>(max_stream, std::max<uint64_t>(1 << 16, std::max<uint64_t>(in_bytes / 8, c->ucap_hint)));
            } else {
                ai.cells = 2 * geo.W; ai.n_words = geo.W;
                const uint64_t guess = 3 * (job.max_row_bytes * 19 / 10) + in_bytes / 100;
                ai.ucap_guess = std::min<uint64_t>(max_stream, std::max<uint64_t>(1 << 16, std::min<uint64_t>(max_stream / 4, std::max<uint64_t>(guess, c->ucap_hint))));
            }
            bool retry = false;
            auto upstream = [&](const uint64_t* s) -> int {
                if (regions && s[S_OVERFLOW]) return 1;
                if (s[S_WU_NEEDED] > wcap) { wcap = s[S_WU_NEEDED] + s[S_WU_NEEDED] / 4 + 4096; again = true; return 1; }
                if (!wide_exact && s[S_WIDE_OVERFLOW]) { wide_exact = true; again = true; c->stats.n_region_overflows++; return 1; }
                return 0;
            };
            const int ar = run_aggregate(c, geo, ai, out, retry, upstream);
            if (ar) return ar;
            if (regions && sc[S_OVERFLOW]) break;
        }   // round
        const bool redo = regions && (sc[S_OVERFLOW] || unit_overflow);
        if (!redo) {
            c->wide_hint = sc[S_N_WIDE];
            if (job.agg != AGG_ROUND) c->ucap_hint = sc[S_U_NEEDED] + sc[S_U_NEEDED] / 8;
            break;
        }
        c->stats.n_region_overflows++;
    }
    if (c->ev_ok && !out.ordered) cudaEventRecord(c->ev[T_AGG], st);
    return GRMKM_OK;
}

// After the aggregate of a final / partial build: bucket chunks -> result arrays (unordered emission), or the chunk
// offsets of a partial build.  Ends with the build's last synchronisation.
int finish_columns(grmkm_ctx* c, const Geo& geo, uint32_t n_words, bool partial, JobOut& out) {
    cudaStream_t st = c->stream;
    uint64_t* d_scalars = (uint64_t*)c->scalars.p;
    const uint64_t U = out.sc[S_U_NEEDED];
    const uint32_t VB = geo.VB;
    if (!out.ordered) {
        ENSURE(c, c->offsets2, (size_t)(VB + 1) * 8);
        ENSURE(c, c->kmers, U * 8);
        ENSURE(c, c->matrix, (size_t)U * n_words * 8);
        k_bucket_offsets<<<1, 1024, 0, st>>>((unsigned long long*)c->bcounts.p, (unsigned long long*)c->offsets2.p, VB,
                                             d_scalars, S_N_SOLID, 1);
        out.launches++;
        if (U && !partial) {
            k_gather_buckets<<<std::min<uint32_t>(VB, (uint32_t)c->sm_count * 8), 256, 0, st>>>(
                (const unsigned long long*)c->ukeys.p, (const unsigned long long*)c->uwords.p, out.ucap,
                (const unsigned long long*)c->bbase.p, (const unsigned long long*)c->offsets2.p, VB, n_words, U,
                (unsigned long long*)c->kmers.p, (unsigned long long*)c->matrix.p, U);
            out.launches++;
        }                               // partial build: grmkm_export_partials gathers straight into the caller's AoS buffer
        CU_TRY(c, cudaGetLastError());
        if (partial) {
            out.h_off.resize(VB + 1);
            CU_TRY(c, cudaMemcpyAsync(out.h_off.data(), c->offsets2.p, (size_t)(VB + 1) * 8, cudaMemcpyDeviceToHost, st));
        }
    }
    c->pitch = out.ordered ? out.ucap : U;
    if (c->ev_ok) cudaEventRecord(c->ev[T_SORT], st);
    CU_TRY(c, cudaStreamSynchronize(st));
    return GRMKM_OK;
}

void add_job_stats(grmkm_ctx* c, const JobOut& o, bool counts_are_final) {
    grmkm_stats& s = c->stats;
    s.n_records += o.sc[S_N_RECORDS];
    s.n_bases += o.sc[S_STREAM_TOTAL] - o.sc[S_N_RECORDS];
    s.n_windows += o.sc[S_N_WINDOWS];
    s.n_launches += o.launches;
    s.h2d_bytes += o.h2d;
    s.n_splits += o.sc[S_N_SPLITS];
    s.n_units += o.sc[S_N_UNITS];
    s.n_unit_entries += o.sc[S_WU_NEEDED];
    s.n_wide += o.sc[S_N_WIDE];
    s.n_unit_buckets = std::max(s.n_unit_buckets, o.MB);
    if (counts_are_final) { s.n_kmers = o.sc[S_U_NEEDED]; s.n_distinct = o.sc[S_N_DISTINCT]; }
}

void set_partial_state(grmkm_ctx* c, const Geo& geo, uint32_t n_ranges, const JobOut& o) {
    // partial columns are in bucket order: owner r holds buckets [r*B/P, (r+1)*B/P)
    c->part_ranks = n_ranges;
    c->part_counts.resize(n_ranges);
    for (uint32_t r = 0; r < n_ranges; ++r)
        c->part_counts[r] = o.h_off[((uint64_t)geo.B * (r + 1) / n_ranges) << geo.sub_bits] - o.h_off[((uint64_t)geo.B * r / n_ranges) << geo.sub_bits];
    c->part_total = o.sc[S_U_NEEDED]; c->part_cap = o.ucap; c->part_buckets = geo.VB;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// the build
// ------------------------------------------------------------------------------------------------
static int merge_sources(grmkm_ctx* c, const void* dev_parts, uint32_t n_ranks, const uint64_t* src_counts, const uint32_t* src_words,
                         uint32_t total_genomes, uint32_t ob, uint64_t own_lo, uint64_t own_hi, uint32_t owners, bool partial_out,
                         bool inside_build);

// ---- presence build of more than 256 genomes: row blocks.  A table slot of the column aggregate holds all the word rows of
// a column, so with many word rows the tables hold few k-mers and split all the time (1,000 genomes on one B200: 10 k
// splits, 62 ms).  Instead the rows are built in blocks of 256 (4 word rows: one dedupe entry / wide record per unit),
// each block leaving sorted partial columns [hash, its words], and the blocks are merged like the ranks of a multi-GPU
// build: k_aggregate_cols<3> keeps one entry REFERENCE per block in its table (10 + 4 x blocks bytes per slot).
static int build_row_blocks(grmkm_ctx* c, const Geo& geo, const InputTable& tab, uint32_t mode, uint32_t n_ranges) {
    cudaStream_t st = c->stream;
    const uint32_t rows_per = kBlockRows * ((geo.W + 4 * 16 - 1) / (4 * 16));          // at most 16 blocks
    const uint32_t R = (geo.G + rows_per - 1) / rows_per;
    std::vector<uint64_t> cnt(R, 0);
    std::vector<uint32_t> words(R, 0);
    uint64_t used = 0;                                  // u64 words of c->racc in use
    ENSURE(c, c->racc, std::max<uint64_t>(1 << 20, c->racc_hint * 8));
    for (uint32_t r = 0; r < R; ++r) {
        const uint32_t row0 = r * rows_per, n_rows = std::min(rows_per, geo.G - row0);
        Geo gr = geo; gr.G = n_rows; gr.W = (n_rows + 63) / 64;
        words[r] = gr.W;
        Job job; job.f0 = tab.first_file[row0]; job.f1 = tab.first_file[row0 + n_rows]; job.row0 = row0; job.n_rows = n_rows;
        job.agg = AGG_PARTIAL;
        for (uint32_t g = row0; g < row0 + n_rows; ++g) job.max_row_bytes = std::max(job.max_row_bytes, tab.row_bytes[g]);
        if (job.f0 == job.f1) continue;
        JobOut out;
        int rc = run_job(c, gr, job, out);
        if (rc) return rc;
        rc = finish_columns(c, gr, gr.W, true, out);
        if (rc) return rc;
        const uint64_t U = out.sc[S_U_NEEDED], need = used + U * (1 + gr.W);
        if (need * 8 > c->racc.cap) {
            DevBuf bigger;
            ENSURE(c, bigger, (need + need / 2) * 8 * (R - r > 1 ? 2 : 1));
            if (used) CU_TRY(c, cudaMemcpyAsync(bigger.p, c->racc.p, used * 8, cudaMemcpyDeviceToDevice, st));
            CU_TRY(c, cudaStreamSynchronize(st));
            release(c, c->racc);
            c->racc = bigger;
        }
        if (U) {
            k_gather_buckets_aos<<<std::min<uint32_t>(gr.VB, (uint32_t)c->sm_count * 8), 256, 0, st>>>(
                (const unsigned long long*)c->ukeys.p, (const unsigned long long*)c->uwords.p, out.ucap,
                (const unsigned long long*)c->bbase.p, (const unsigned long long*)c->offsets2.p, gr.VB, gr.W,
                (unsigned long long*)c->racc.p + used);
            out.launches++;
            CU_TRY(c, cudaGetLastError());
        }
        cnt[r] = U; used = need;
        add_job_stats(c, out, false);
        add_stage_times(c);
    }
    c->racc_hint = used + used / 8;
    const uint32_t ob = mode == 1 ? geo.bucket_bits : 0u;
    int rc = merge_sources(c, c->racc.p, R, cnt.data(), words.data(), geo.G, ob, 0, 1ULL << ob, 1, mode == 1, true);
    if (rc) return rc;
    c->stats.n_buckets = geo.B; c->stats.device_bytes = c->device_bytes; c->stats.n_rounds = R;
    c->stats.n_genomes = geo.G; c->stats.n_words = geo.W;
    if (mode == 1) {
        // the merged partial columns are bucket chunks on the merge grid (2^merge_bits >= 2^bucket_bits buckets)
        const uint32_t sub = c->merge_bits > geo.bucket_bits ? c->merge_bits - geo.bucket_bits : 0u;
        c->part_ranks = n_ranges;
        c->part_counts.assign(n_ranges, 0);
        if (c->merge_h_off.size() > 2)
            for (uint32_t r = 0; r < n_ranges; ++r)
                c->part_counts[r] = c->merge_h_off[((uint64_t)geo.B * (r + 1) / n_ranges) << sub] - c->merge_h_off[((uint64_t)geo.B * r / n_ranges) << sub];
        c->part_total = c->U; c->part_cap = c->merge_cap; c->part_buckets = c->merge_bits ? (1u << c->merge_bits) : geo.B;
        c->part_words = geo.W;
        c->built = false;
    }
    return GRMKM_OK;
}

static int build_impl(grmkm_ctx* c, uint32_t mode /*0 final, 1 partial*/, uint32_t n_ranges) {
    CU_TRY(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    c->built = false;
    c->stats = grmkm_stats{};
    c->times = grmkm_times{};

    const bool pooled = (c->cfg.flags & GRMKM_FLAG_COUNTS) != 0;
    if (pooled) {
        if (mode == 1) return fail(c, GRMKM_E_UNSUPPORTED, "the pooled count table is a one-GPU build");
        for (Input& in : c->inputs) in.row = 0;              // dsk -file <list>: every file is pooled (src/app.py:1371-1372)
        c->n_genomes_decl = std::min(c->n_genomes_decl, 1u);
    }
    const InputTable tab = tabulate_inputs(c);
    Geo geo;
    geo.G = tab.G; geo.W = (tab.G + 63) / 64;
    const uint32_t F = (uint32_t)c->inputs.size();
    c->G = geo.G; c->W = geo.W; c->U = 0;
    c->part_ranks = 0; c->part_total = 0; c->part_words = geo.W;
    c->stats.n_genomes = geo.G; c->stats.n_words = geo.W; c->stats.n_input_bytes = tab.in_bytes;
    if (geo.G == 0 || F == 0) {
        c->built = (mode == 0);
        if (mode == 1) { c->part_ranks = n_ranges; c->part_counts.assign(n_ranges, 0); }
        return GRMKM_OK;
    }
    if (geo.G > 32768) return fail(c, GRMKM_E_UNSUPPORTED, "more than 32768 genomes in one context");

    // ---- bucket count.  The expansion sorts tiles over at most 2^11 buckets: more distinct k-mers than 2^11 tables
    // hold are handled as key sub-ranges of the buckets (virtual buckets: one aggregate pass each over the bucket's
    // records, which stay in L2), and beyond 2^14 by the table's own overflow split.
    uint32_t bits = c->cfg.bucket_bits ? c->cfg.bucket_bits : auto_bucket_bits(c, tab);
    // the records' group field replaces bucket bits; a partial build keeps the agreed count as it is (every rank must
    // cut the hash space the same way whatever its share of the rows)
    if (mode == 0) bits = std::max(bits, std::max(1u, ceil_log2(geo.W)));
    if (bits > 15) return fail(c, GRMKM_E_UNSUPPORTED, "bucket_bits > 15");
    if (const char* sbv = getenv("GRMKM_SUB_BITS")) geo.sub_bits = (uint32_t)std::min(3, std::max(0, atoi(sbv)));
    if (bits > kUnitMaxBucketBits) {
        geo.sub_bits = std::max(geo.sub_bits, std::min(kMaxSubBits, bits - kUnitMaxBucketBits));
        bits = kUnitMaxBucketBits;
    }
    geo.bucket_bits = bits; geo.B = 1u << bits; geo.VB = geo.B << geo.sub_bits;
    c->cur_bucket_bits = bits;

    if (!abundance_build(c) && geo.G > kBlockRows && !getenv("GRMKM_NO_ROW_BLOCKS")) return build_row_blocks(c, geo, tab, mode, n_ranges);
    if (!abundance_build(c)) {
        // ---- presence build (contigs, reads without an abundance filter): one pass over everything
        Job job; job.f0 = 0; job.f1 = F; job.row0 = 0; job.n_rows = geo.G; job.max_row_bytes = tab.max_row;
        job.agg = mode == 0 ? AGG_FINAL : AGG_PARTIAL;
        JobOut out;
        int r = run_job(c, geo, job, out);
        if (r) return r;
        r = finish_columns(c, geo, geo.W, mode == 1, out);
        if (r) return r;
        add_job_stats(c, out, true);
        add_stage_times(c);
        c->stats.n_buckets = geo.B; c->stats.device_bytes = c->device_bytes;
        c->U = out.sc[S_U_NEEDED];
        c->built = (mode == 0);
        if (mode == 1) set_partial_state(c, geo, n_ranges, out);
        return GRMKM_OK;
    }

    if (pooled) {
        // ---- pooled count table (dsk): one round, the aggregate emits (k-mer, count) columns
        Job job; job.f0 = 0; job.f1 = F; job.row0 = 0; job.n_rows = 1; job.max_row_bytes = tab.in_bytes; job.agg = AGG_COUNTS;
        JobOut out;
        int r = run_job(c, geo, job, out);
        if (r) return r;
        r = finish_columns(c, geo, 1, false, out);
        if (r) return r;
        add_job_stats(c, out, true);
        add_stage_times(c);
        c->stats.n_buckets = geo.B; c->stats.device_bytes = c->device_bytes;
        c->U = out.sc[S_U_NEEDED];
        c->built = true;
        return GRMKM_OK;
    }

    // ---- abundance build (reads with -abundance-min > 1): rounds of a few genome rows, each leaving the solid
    // presence of its rows as records [(hash << wbits) | matrix word, bits]; then ONE presence aggregate over the
    // records of all rounds.
    const std::vector<Round> rounds = plan_rounds(c, geo.G, tab.first_file, tab.row_bytes);
    struct Seg { unsigned long long src, dst, n; };
    std::vector<std::vector<uint64_t>> r_base(rounds.size()), r_cnt(rounds.size());
    uint64_t used = 0;
    {
        // one record per solid (k-mer, round): about the text's 64th part for read sets; the buffer doubles when a round
        // does not fit
        const uint64_t guess = std::max<uint64_t>(1 << 16, std::max<uint64_t>(tab.in_bytes / 64, c->racc_hint));
        ENSURE(c, c->racc, guess * 16);
    }
    for (size_t ri = 0; ri < rounds.size(); ++ri) {
        const Round& rd = rounds[ri];
        r_base[ri].assign(geo.VB, 0); r_cnt[ri].assign(geo.VB, 0);
        if (rd.f1 == rd.f0) continue;                      // rows without input
        Job job; job.f0 = rd.f0; job.f1 = rd.f1; job.row0 = rd.row0; job.n_rows = rd.n_rows; job.agg = AGG_ROUND;
        for (uint32_t g = rd.row0; g < rd.row0 + rd.n_rows; ++g) job.max_row_bytes = std::max(job.max_row_bytes, tab.row_bytes[g]);
        for (int attempt = 0;; ++attempt) {
            job.round_out = (ulonglong2*)c->racc.p + used;
            job.round_cap = c->racc.cap / 16 - used;
            JobOut out;
            int r = run_job(c, geo, job, out);
            if (r) return r;
            if (c->ev_ok) cudaEventRecord(c->ev[T_SORT], st);
            if (out.round_full) {
                if (attempt > 2) return fail(c, GRMKM_E_NOMEM, "abundance round output does not fit");
                // grow: what is there + this round's need, doubled for the rounds to come
                const uint64_t want = (used + out.sc[S_U_NEEDED]) * 2 + 4096;
                DevBuf bigger;
                ENSURE(c, bigger, want * 16);
                if (used) CU_TRY(c, cudaMemcpyAsync(bigger.p, c->racc.p, used * 16, cudaMemcpyDeviceToDevice, st));
                CU_TRY(c, cudaStreamSynchronize(st));
                release(c, c->racc);
                c->racc = bigger;
                c->stats.n_launches += out.launches;
                continue;
            }
            CU_TRY(c, cudaMemcpyAsync(r_base[ri].data(), c->bbase.p, (size_t)geo.VB * 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(c, cudaMemcpyAsync(r_cnt[ri].data(), c->bcounts.p, (size_t)geo.VB * 8, cudaMemcpyDeviceToHost, st));
            CU_TRY(c, cudaStreamSynchronize(st));
            for (uint32_t v = 0; v < geo.VB; ++v) r_base[ri][v] += used;       // the aggregate counts from its own output pointer
            used += out.sc[S_U_NEEDED];
            add_job_stats(c, out, false);
            add_stage_times(c);
            break;
        }
    }
    c->racc_hint = used + used / 8;
    // ---- records of all rounds, bucket by bucket (exact offsets), then the presence aggregate
    std::vector<Seg> segs;
    std::vector<uint64_t> h_begin(geo.B + 1, 0);
    {
        uint64_t pos = 0;
        for (uint32_t v = 0; v < geo.VB; ++v) {
            if ((v & ((1u << geo.sub_bits) - 1u)) == 0) h_begin[v >> geo.sub_bits] = pos;
            for (size_t ri = 0; ri < rounds.size(); ++ri)
                if (r_cnt[ri][v]) { segs.push_back(Seg{r_base[ri][v], pos, r_cnt[ri][v]}); pos += r_cnt[ri][v]; }
        }
        h_begin[geo.B] = pos;
    }
    JobOut out;
    ENSURE(c, c->scalars, S_COUNT * 8);
    ENSURE(c, c->offsets, (size_t)(geo.B + 1) * 8);
    ENSURE(c, c->wide, (used + 1) * 16);
    ENSURE(c, c->refs, std::max<size_t>(1, segs.size()) * sizeof(Seg));
    uint64_t* d_scalars = (uint64_t*)c->scalars.p;
    if (c->ev_ok) for (int e = T_START; e < T_AGG; ++e) cudaEventRecord(c->ev[e], st);
    CU_TRY(c, cudaMemsetAsync(d_scalars, 0, S_COUNT * 8, st));
    CU_TRY(c, cudaMemcpyAsync(c->offsets.p, h_begin.data(), (size_t)(geo.B + 1) * 8, cudaMemcpyHostToDevice, st));
    if (!segs.empty()) {
        CU_TRY(c, cudaMemcpyAsync(c->refs.p, segs.data(), segs.size() * sizeof(Seg), cudaMemcpyHostToDevice, st));
        k_gather_segments<<<(uint32_t)std::min<size_t>(segs.size(), (size_t)c->sm_count * 16), 128, 0, st>>>(
            (const ulonglong2*)c->racc.p, (const unsigned long long*)c->refs.p, (uint32_t)segs.size(), (ulonglong2*)c->wide.p);
        out.launches++;
        CU_TRY(c, cudaGetLastError());
    }
    if (c->ev_ok) cudaEventRecord(c->ev[T_EXPAND], st);
    AggIn ai{};
    ai.records = (const unsigned long long*)c->wide.p;
    ai.begin = (const unsigned long long*)c->offsets.p; ai.end = ai.begin + 1;
    ai.wide_words = 1; ai.wide_stride = 2; ai.row_bits = std::max(1u, ceil_log2(geo.W));
    ai.cells = 2 * geo.W; ai.n_words = geo.W; ai.agg = mode == 0 ? AGG_FINAL : AGG_PARTIAL;
    ai.ucap_guess = std::max<uint64_t>(1 << 12, std::min<uint64_t>(used, std::max<uint64_t>(c->ucap_hint, used / 2)));
    bool retry = false;
    int r = run_aggregate(c, geo, ai, out, retry, [](const uint64_t*) { return 0; });
    if (r) return r;
    if (c->ev_ok && !out.ordered) cudaEventRecord(c->ev[T_AGG], st);
    c->ucap_hint = out.sc[S_U_NEEDED] + out.sc[S_U_NEEDED] / 8;
    r = finish_columns(c, geo, geo.W, mode == 1, out);
    if (r) return r;
    c->stats.n_launches += out.launches;
    c->stats.n_kmers = out.sc[S_U_NEEDED]; c->stats.n_distinct = out.sc[S_N_DISTINCT]; c->stats.n_splits += out.sc[S_N_SPLITS];
    c->stats.n_solid_records = used; c->stats.n_rounds = (uint32_t)rounds.size();
    add_stage_times(c);
    c->stats.n_buckets = geo.B; c->stats.device_bytes = c->device_bytes;
    c->U = out.sc[S_U_NEEDED];
    c->built = (mode == 0);
    if (mode == 1) set_partial_state(c, geo, n_ranges, out);
    return GRMKM_OK;
}

// What described the last result goes with it: its slice flag, pattern multiplicities and learners' results (all that
// goes in the owner-side merge of a multi-GPU build, which sets built itself and keeps the partial state it merged)
static void forget_result(grmkm_ctx* c) {
    c->slice = false;
    c->pat_mult_on = false;
    c->scm_steps.clear(); c->scm_equiv.clear();
    c->cart_nodes.clear(); c->cart_equiv.clear();
}

// A result replaces the last one.  built: the U x W matrix over G genomes in place is whole (patterns: a pattern matrix),
// and the stats and times restart from it; else there is none, whole or partial (a reset, a build until it succeeds).
static void set_result(grmkm_ctx* c, bool built, bool patterns = false) {
    forget_result(c);
    c->built = built;
    c->part_ranks = 0;
    c->pat_mult_on = patterns;
    if (!built) return;
    c->stats = grmkm_stats{};
    c->stats.n_kmers = c->stats.n_distinct = c->U;
    c->stats.n_words = c->W; c->stats.n_genomes = c->G;
    c->times = grmkm_times{};
}

// every failure of a build leaves the context quiet: nothing in flight reads borrowed host buffers any more, and no
// side-stream clear is counted on
static int build_guarded(grmkm_ctx* c, uint32_t mode, uint32_t n_ranges) {
    NvtxRange nv(mode == 0 ? "grmkm_build" : "grmkm_build_partial");
    set_result(c, false);
    const int r = build_impl(c, mode, n_ranges);
    if (r != GRMKM_OK) {
        const std::string msg = c->err;
        cudaStreamSynchronize(c->stream);
        if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
        if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);
        cudaGetLastError();
        c->pre_pending = false;
        set_result(c, false);
        c->err = msg;
    }
    return r;
}

extern "C" {

int grmkm_abi_version(void) { return GRMKM_ABI_VERSION; }

int grmkm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int grmkm_create(const grmkm_config* cfg, grmkm_ctx** out) {
    if (!cfg || !out) return fail(nullptr, GRMKM_E_INVALID, "null argument");
    *out = nullptr;
    grmkm_config c{};
    memcpy(&c, cfg, std::min<size_t>(sizeof c, cfg->struct_size ? cfg->struct_size : sizeof c));
    if (c.k < 1 || c.k > 32)
        return fail(nullptr, GRMKM_E_UNSUPPORTED_K, "k must be in 1..32 (got " + std::to_string(c.k) + ")");
    if (c.min_abundance == 0) c.min_abundance = 1;
    if (c.input_kind > GRMKM_FASTQ) return fail(nullptr, GRMKM_E_INVALID, "input_kind must be GRMKM_FASTA or GRMKM_FASTQ");
    if (c.flags & ~GRMKM_FLAG_COUNTS) return fail(nullptr, GRMKM_E_INVALID, "unknown flag bits");
    if (c.bucket_bits && (c.bucket_bits < 4 || c.bucket_bits > 15))
        return fail(nullptr, GRMKM_E_INVALID, "bucket_bits must be 0 (auto) or 4..15");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, GRMKM_E_NO_DEVICE,
                    std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "0 devices") +
                        "); libgrmkm has no CPU fallback");
    }
    int dev = c.device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= ndev) return fail(nullptr, GRMKM_E_INVALID, "device ordinal out of range");
    if ((e = cudaSetDevice(dev)) != cudaSuccess)
        return fail(nullptr, GRMKM_E_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    grmkm_ctx* x = new (std::nothrow) grmkm_ctx();
    if (!x) return fail(nullptr, GRMKM_E_NOMEM, "out of host memory");
    x->cfg = c;
    x->device = dev;
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
        x->sm_count = prop.multiProcessorCount;
        x->smem_optin = prop.sharedMemPerBlockOptin;
    }
    if (const char* bb = getenv("GRMKM_BATCH_BYTES")) { const long long v = atoll(bb); if (v > 0) x->batch_bytes = (uint64_t)v; }
    if (c.stream) x->stream = (cudaStream_t)c.stream;
    else {
        if ((e = cudaStreamCreateWithFlags(&x->stream, cudaStreamNonBlocking)) != cudaSuccess) {
            delete x;
            return fail(nullptr, GRMKM_E_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
        }
        x->own_stream = true;
    }
    x->ev_ok = true;
    for (int i = 0; i < T_N; ++i) {
        if (cudaEventCreate(&x->ev[i]) != cudaSuccess) {
            // no stage timing then; the events that were created are not kept
            cudaGetLastError();
            for (int j = 0; j < i; ++j) cudaEventDestroy(x->ev[j]);
            x->ev_ok = false;
            break;
        }
    }
    *out = x;
    return GRMKM_OK;
}

void grmkm_destroy(grmkm_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);      // the clear for a next build may still be running
    DevBuf* all[] = {&c->in, &c->files, &c->hdr0, &c->tile_file, &c->tile_pub, &c->tile_order,
                     &c->fss, &c->codes, &c->valid, &c->hist, &c->offsets, &c->offsets2,
                     &c->bcounts, &c->ukeys, &c->uwords, &c->kmers, &c->matrix, &c->scalars, &c->fmt, &c->synth, &c->refs,
                     &c->stile_file, &c->bbase, &c->apub, &c->masks, &c->units, &c->ucur, &c->ubeg, &c->wu, &c->wide,
                     &c->racc, &c->aux, &c->scm, &c->scm_list, &c->cart, &c->cart_bl,
                     &c->cart_masks[0], &c->cart_masks[1], &c->cart_list, &c->qry, &c->qplane, &c->qout, &c->eval,
                     &c->shard_idx, &c->shard_cols};
    for (DevBuf* b : all) release(c, *b);
    if (c->ev_ok) for (int i = 0; i < T_N; ++i) cudaEventDestroy(c->ev[i]);
    for (cudaEvent_t e : c->ev_query) if (e) cudaEventDestroy(e);
    if (c->host_res) cudaFreeHost(c->host_res);
    if (c->aux_stream) {
        cudaEventDestroy(c->ev_scattered); cudaEventDestroy(c->ev_cleared);
        cudaStreamDestroy(c->aux_stream);
    }
    if (c->copy_stream) {
        for (int i = 0; i < 2; ++i) { cudaEventDestroy(c->ev_copied[i]); cudaEventDestroy(c->ev_free[i]); }
        cudaStreamDestroy(c->copy_stream);
    }
    if (c->h_tab) cudaFreeHost(c->h_tab);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* grmkm_last_error(const grmkm_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int grmkm_reset(grmkm_ctx* c) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    c->inputs.clear();
    c->n_genomes_decl = 0;
    c->U = 0; c->W = 0; c->G = 0;
    set_result(c, false);
    return GRMKM_OK;
}

int grmkm_add_genome_bytes(grmkm_ctx* c, uint32_t row, const uint8_t* data, uint64_t n) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!data && n) return fail(c, GRMKM_E_INVALID, "null data");
    if (row >= kMaxGenomes) return fail(c, GRMKM_E_UNSUPPORTED, "genome row out of range (at most 32768 genomes in one context)");
    Input in; in.row = row; in.kind = c->cfg.input_kind; in.host = data; in.len = n;
    c->inputs.push_back(std::move(in));
    c->built = false;
    return GRMKM_OK;
}

int grmkm_add_genome_device(grmkm_ctx* c, uint32_t row, const void* dev_data, uint64_t n) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!dev_data && n) return fail(c, GRMKM_E_INVALID, "null data");
    if ((uintptr_t)dev_data & 15) return fail(c, GRMKM_E_INVALID, "device input must be 16-byte aligned");
    if (row >= kMaxGenomes) return fail(c, GRMKM_E_UNSUPPORTED, "genome row out of range (at most 32768 genomes in one context)");
    Input in; in.row = row; in.kind = c->cfg.input_kind; in.dev = (const uint8_t*)dev_data; in.len = n;
    c->inputs.push_back(std::move(in));
    c->built = false;
    return GRMKM_OK;
}

int grmkm_add_genomes(grmkm_ctx* c, uint32_t n, const uint32_t* rows, const void* const* data, const uint64_t* lens,
                      int on_device) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (n && (!rows || !data || !lens)) return fail(c, GRMKM_E_INVALID, "null input list");
    c->inputs.reserve(c->inputs.size() + n);
    for (uint32_t i = 0; i < n; ++i) {
        const int r = on_device ? grmkm_add_genome_device(c, rows[i], data[i], lens[i])
                                : grmkm_add_genome_bytes(c, rows[i], (const uint8_t*)data[i], lens[i]);
        if (r) return r;
    }
    return GRMKM_OK;
}

int grmkm_add_genome_files(grmkm_ctx* c, uint32_t row, const char* const* paths, int n_paths) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (n_paths < 0 || (!paths && n_paths)) return fail(c, GRMKM_E_INVALID, "bad path list");
    if (row >= kMaxGenomes) return fail(c, GRMKM_E_UNSUPPORTED, "genome row out of range (at most 32768 genomes in one context)");
    for (int i = 0; i < n_paths; ++i) {
        Input in; in.row = row; in.kind = c->cfg.input_kind;
        int r = read_file(c, paths[i], in.owned);
        if (r) return r;
        in.len = in.owned.size();
        c->inputs.push_back(std::move(in));
        c->inputs.back().host = c->inputs.back().owned.data();
    }
    c->built = false;
    return GRMKM_OK;
}

int grmkm_set_genome_count(grmkm_ctx* c, uint32_t n) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (n > kMaxGenomes) return fail(c, GRMKM_E_UNSUPPORTED, "at most 32768 genomes in one context");
    c->n_genomes_decl = n;
    return GRMKM_OK;
}


int grmkm_build(grmkm_ctx* c) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    return build_guarded(c, 0, 1);
}

int grmkm_dims(const grmkm_ctx* c, uint64_t* n_kmers, uint32_t* n_words, uint32_t* n_genomes) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(const_cast<grmkm_ctx*>(c), GRMKM_E_INVALID, "no result: call grmkm_build first");
    if (n_kmers) *n_kmers = c->U;
    if (n_words) *n_words = c->W;
    if (n_genomes) *n_genomes = c->G;
    return GRMKM_OK;
}

int grmkm_get_stats(const grmkm_ctx* c, grmkm_stats* out) {
    if (check_ctx(c) || !out) return GRMKM_E_INVALID;
    *out = c->stats;
    out->device_bytes = c->device_bytes;
    return GRMKM_OK;
}

int grmkm_stage_times(const grmkm_ctx* c, grmkm_times* out) {
    if (check_ctx(c) || !out) return GRMKM_E_INVALID;
    *out = c->times;
    return GRMKM_OK;
}

int grmkm_copy_kmers_packed(grmkm_ctx* c, uint64_t* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    if (cap < c->U) return fail(c, GRMKM_E_CAPACITY, "kmers buffer too small");
    if (!c->U) return GRMKM_OK;
    if (!dst) return fail(c, GRMKM_E_INVALID, "null dst");
    CU_TRY(c, cudaSetDevice(c->device));
    CU_TRY(c, cudaMemcpyAsync(dst, c->kmers.p, c->U * 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_copy_matrix(grmkm_ctx* c, uint64_t* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    const uint64_t n = c->U * c->W;
    if (cap < n) return fail(c, GRMKM_E_CAPACITY, "matrix buffer too small");
    if (!n) return GRMKM_OK;
    if (!dst) return fail(c, GRMKM_E_INVALID, "null dst");
    CU_TRY(c, cudaSetDevice(c->device));
    // (rows are c->pitch words apart on the device, U words apart in the caller's array)
    CU_TRY(c, cudaMemcpy2DAsync(dst, c->U * 8, c->matrix.p, c->pitch * 8, c->U * 8, c->W, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_copy_kmer_strings(grmkm_ctx* c, char* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    const uint32_t k = c->cfg.k;
    const uint64_t n = c->U * k;
    if (cap < n) return fail(c, GRMKM_E_CAPACITY, "kmer string buffer too small");
    if (!n) return GRMKM_OK;
    if (!dst) return fail(c, GRMKM_E_INVALID, "null dst");
    CU_TRY(c, cudaSetDevice(c->device));
    const uint64_t rows_per = std::max<uint64_t>(1, (256ULL << 20) / k);
    ENSURE(c, c->fmt, std::min<uint64_t>(n, rows_per * k));
    for (uint64_t j0 = 0; j0 < c->U; j0 += rows_per) {
        const uint64_t rows = std::min(rows_per, c->U - j0), nb = rows * k;
        k_kmer_strings<<<(uint32_t)((nb + 255) / 256), 256, 0, c->stream>>>((const unsigned long long*)c->kmers.p, j0, nb,
                                                                            k, (char*)c->fmt.p);
        CU_TRY(c, cudaGetLastError());
        CU_TRY(c, cudaMemcpyAsync(dst + j0 * k, c->fmt.p, nb, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
    }
    return GRMKM_OK;
}

int grmkm_format_tsv(grmkm_ctx* c, const char* const* names, char* dst, uint64_t cap, uint64_t* written) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    if (!names && c->G) return fail(c, GRMKM_E_INVALID, "null names");
    const uint32_t k = c->cfg.k, G = c->G;
    uint64_t hdr = 5;
    for (uint32_t g = 0; g < G; ++g) {
        if (!names[g]) return fail(c, GRMKM_E_INVALID, "null name");
        hdr += 1 + strlen(names[g]);
    }
    hdr += 1;
    const uint64_t roww = (uint64_t)k + 2ULL * G + 1;
    const uint64_t need = hdr + roww * c->U;
    if (written) *written = need;
    if (!dst || cap < need) return fail(c, GRMKM_E_CAPACITY, "tsv buffer too small");
    char* p = dst;
    memcpy(p, "kmers", 5); p += 5;
    for (uint32_t g = 0; g < G; ++g) { *p++ = '\t'; size_t l = strlen(names[g]); memcpy(p, names[g], l); p += l; }
    *p++ = '\n';
    if (!c->U) return GRMKM_OK;
    CU_TRY(c, cudaSetDevice(c->device));
    const uint64_t rows_per = std::max<uint64_t>(1, (256ULL << 20) / roww);
    ENSURE(c, c->fmt, std::min<uint64_t>(roww * c->U, rows_per * roww));
    for (uint64_t j0 = 0; j0 < c->U; j0 += rows_per) {
        const uint64_t rows = std::min(rows_per, c->U - j0), nb = rows * roww;
        k_format_tsv<<<(uint32_t)((nb + 255) / 256), 256, 0, c->stream>>>((const unsigned long long*)c->kmers.p,
                                                                          (const unsigned long long*)c->matrix.p, c->pitch, G,
                                                                          k, j0, nb, (char*)c->fmt.p);
        CU_TRY(c, cudaGetLastError());
        CU_TRY(c, cudaMemcpyAsync(p + j0 * roww, c->fmt.p, nb, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
    }
    return GRMKM_OK;
}

int grmkm_host_result(grmkm_ctx* c, const uint64_t** kmers, const uint64_t** matrix) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    const size_t nk = (size_t)c->U * 8, nm = (size_t)c->U * c->W * 8;
    CU_TRY(c, cudaSetDevice(c->device));
    if (c->host_res_cap < nk + nm + 16) {
        if (c->host_res) { cudaFreeHost(c->host_res); c->host_res = nullptr; c->host_res_cap = 0; }
        const size_t want = ((nk + nm) * 5 / 4 + (1 << 20)) & ~size_t(4095);
        cudaError_t e = cudaHostAlloc(&c->host_res, want, cudaHostAllocDefault);
        if (e != cudaSuccess) { c->host_res = nullptr; return fail(c, GRMKM_E_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
        c->host_res_cap = want;
    }
    uint8_t* h = (uint8_t*)c->host_res;
    NvtxRange nv("grmkm_host_result: device -> host");
    // In pieces of 4 MiB: a single large device->host copy starves the host->device copies of another context that is
    // staging its text at the same time (BuildPipeline); in pieces both directions keep moving
    // (profiles/r02_duplex_pattern.txt).  Rows are c->pitch words apart on the device, U words apart on the host.
    constexpr size_t kPiece = 4u << 20;
    for (size_t o = 0; o < nk; o += kPiece)
        CU_TRY(c, cudaMemcpyAsync(h + o, (const uint8_t*)c->kmers.p + o, std::min(kPiece, nk - o), cudaMemcpyDeviceToHost, c->stream));
    for (uint32_t w = 0; w < c->W && nm; ++w)
        for (size_t o = 0; o < nk; o += kPiece)
            CU_TRY(c, cudaMemcpyAsync(h + nk + (size_t)w * nk + o, (const uint8_t*)c->matrix.p + (size_t)w * c->pitch * 8 + o,
                                      std::min(kPiece, nk - o), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    if (kmers) *kmers = (const uint64_t*)h;
    if (matrix) *matrix = (const uint64_t*)(h + nk);
    return GRMKM_OK;
}

int grmkm_device_result(const grmkm_ctx* c, const uint64_t** d_kmers, const uint64_t** d_matrix, uint64_t* pitch_words) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(const_cast<grmkm_ctx*>(c), GRMKM_E_INVALID, "no result: call grmkm_build first");
    if (d_kmers) *d_kmers = (const uint64_t*)c->kmers.p;
    if (d_matrix) *d_matrix = (const uint64_t*)c->matrix.p;
    if (pitch_words) *pitch_words = c->pitch;
    return GRMKM_OK;
}

int grmkm_synth_fasta_device(grmkm_ctx* c, const void* layout, uint64_t layout_bytes, void* dev_dst, uint64_t dst_bytes) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!layout || !dev_dst) return fail(c, GRMKM_E_INVALID, "null argument");
    CU_TRY(c, cudaSetDevice(c->device));
    ENSURE(c, c->synth, layout_bytes);
    CU_TRY(c, cudaMemcpyAsync(c->synth.p, layout, layout_bytes, cudaMemcpyHostToDevice, c->stream));
    std::string msg;
    if (!synth_launch((const uint8_t*)layout, layout_bytes, (const uint8_t*)c->synth.p, (uint8_t*)dev_dst, dst_bytes,
                      c->stream, msg))
        return fail(c, GRMKM_E_INVALID, msg);
    CU_TRY(c, cudaGetLastError());
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_set_bucket_bits(grmkm_ctx* c, uint32_t bits) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (bits && (bits < 4 || bits > 15)) return fail(c, GRMKM_E_INVALID, "bucket_bits must be 0 (auto) or 4..15");
    c->cfg.bucket_bits = bits;
    return GRMKM_OK;
}

int grmkm_set_exchange_rank(grmkm_ctx* c, uint32_t rank) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (rank >= 16) return fail(c, GRMKM_E_INVALID, "rank out of range (at most 16 ranks)");
    c->xrank = (int32_t)rank;
    return GRMKM_OK;
}

int grmkm_plan_bucket_bits(grmkm_ctx* c, uint32_t* bits) {
    if (check_ctx(c) || !bits) return GRMKM_E_INVALID;
    const InputTable tab = tabulate_inputs(c);
    *bits = tab.G ? auto_bucket_bits(c, tab) : 6;
    return GRMKM_OK;
}

int grmkm_build_partial(grmkm_ctx* c, uint32_t n_ranks, uint64_t* counts) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (n_ranks < 1 || n_ranks > 16 || !counts) return fail(c, GRMKM_E_INVALID, "n_ranks must be 1..16");
    if (n_ranks > 1 && !c->cfg.bucket_bits)
        return fail(c, GRMKM_E_INVALID, "the ranks of a multi-GPU build agree on the bucket count first (grmkm_plan_bucket_bits / grmkm_set_bucket_bits)");
    int r = build_guarded(c, 1, n_ranks);
    if (r) return r;
    for (uint32_t i = 0; i < n_ranks; ++i) counts[i] = c->part_counts[i];
    return GRMKM_OK;
}

int grmkm_export_partials(grmkm_ctx* c, void* dev_dst, uint64_t dst_bytes) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->part_ranks) return fail(c, GRMKM_E_INVALID, "no partial result: call grmkm_build_partial first");
    const uint64_t need = c->part_total * (1 + (uint64_t)c->part_words) * 8;
    if (dst_bytes < need) return fail(c, GRMKM_E_CAPACITY, "partial export buffer too small");
    if (!c->part_total) return GRMKM_OK;
    if (!dev_dst) return fail(c, GRMKM_E_INVALID, "null dst");
    CU_TRY(c, cudaSetDevice(c->device));
    k_gather_buckets_aos<<<std::min<uint32_t>(c->part_buckets, (uint32_t)c->sm_count * 8), 256, 0, c->stream>>>(
        (const unsigned long long*)c->ukeys.p, (const unsigned long long*)c->uwords.p, c->part_cap,
        (const unsigned long long*)c->bbase.p, (const unsigned long long*)c->offsets2.p, c->part_buckets, c->part_words,
        (unsigned long long*)dev_dst);
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches++;
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_export_partials_peers(grmkm_ctx* c, uint32_t n_ranks, void* const* peer_dst, const uint64_t* peer_word_off) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->part_ranks) return fail(c, GRMKM_E_INVALID, "no partial result: call grmkm_build_partial first");
    if (n_ranks != c->part_ranks || n_ranks > 16 || !peer_dst || !peer_word_off)
        return fail(c, GRMKM_E_INVALID, "bad peer export arguments");
    if (!c->part_total) return GRMKM_OK;
    CU_TRY(c, cudaSetDevice(c->device));
    PeerSlices ps{};
    ps.n = n_ranks;
    const uint32_t sub = ceil_log2(std::max(1u, c->part_buckets >> c->cur_bucket_bits));      // virtual buckets per bucket
    const uint64_t B = 1ULL << c->cur_bucket_bits;
    for (uint32_t d = 0; d <= n_ranks; ++d) ps.first[d] = (uint32_t)((B * d / n_ranks) << sub);
    ps.rot = ps.first[((uint32_t)(c->xrank >= 0 ? c->xrank : c->device) + 1u) % n_ranks];
    for (uint32_t d = 0; d < n_ranks; ++d) {
        if (c->part_counts[d] && !peer_dst[d]) return fail(c, GRMKM_E_INVALID, "null peer buffer");
        ps.dst[d] = (unsigned long long*)peer_dst[d] + peer_word_off[d];
    }
    k_gather_buckets_peers<<<std::min<uint32_t>(c->part_buckets, (uint32_t)c->sm_count * 8), 256, 0, c->stream>>>(
        (const unsigned long long*)c->ukeys.p, (const unsigned long long*)c->uwords.p, c->part_cap,
        (const unsigned long long*)c->bbase.p, (const unsigned long long*)c->offsets2.p, c->part_buckets, c->part_words, ps);
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches++;
    return GRMKM_OK;             // asynchronous on the context's stream: the caller's barrier follows on the same stream
}

}  // extern "C"

// Merge of n_src lists of partial columns [hash, words...] (each ascending by hash, back to back in dev_parts) into
// columns: the owner-side merge of a multi-GPU build (own_lo .. own_hi of 2^ob = this owner's hash range) and the
// merge of the row blocks of a one-GPU build with more than 256 genomes (the whole hash range).  partial_out: emit
// partial columns again (hash keys, no singleton filter) -- the row blocks of ONE rank of a multi-GPU build.
static int merge_sources(grmkm_ctx* c, const void* dev_parts, uint32_t n_ranks, const uint64_t* src_counts, const uint32_t* src_words,
                         uint32_t total_genomes, uint32_t ob, uint64_t own_lo, uint64_t own_hi, uint32_t owners, bool partial_out,
                         bool inside_build) {
    NvtxRange nv("grmkm merge of sorted partial-column lists");
    cudaStream_t st = c->stream;
    Launches L;
    AggParams2 ap{};
    uint64_t n_total = 0, words = 0;
    uint32_t W_total = 0;
    std::vector<uint64_t> h_meta(3 * 16, 0);          // src_off[16], src_count[16], src_width[16] (as u64 / u32 below)
    uint32_t h_width[16] = {0};
    for (uint32_t s = 0; s < n_ranks; ++s) {
        ap.src_off[s] = words; ap.src_words[s] = src_words[s]; ap.src_woff[s] = W_total;
        h_meta[s] = words; h_meta[16 + s] = src_counts[s]; h_width[s] = 1 + src_words[s];
        n_total += src_counts[s]; words += src_counts[s] * (1 + (uint64_t)src_words[s]); W_total += src_words[s];
    }
    ap.n_src = n_ranks;
    if (W_total != (total_genomes + 63) / 64) return fail(c, GRMKM_E_INVALID, "source words do not add up to the genome count");
    if (n_total && !dev_parts) return fail(c, GRMKM_E_INVALID, "null parts");
    c->built = false; c->U = 0; c->W = W_total; c->G = total_genomes;
    if (!inside_build) c->times = grmkm_times{};
    const uint32_t launches_before = c->stats.n_launches;
    if (n_total == 0) {
        c->built = !partial_out; c->stats.n_kmers = 0;
        if (partial_out) { c->merge_h_off.assign(2, 0); c->merge_bits = 0; c->merge_cap = 0; }
        return GRMKM_OK;
    }
    // the merge table keeps one entry reference per source and slot instead of the words (k_aggregate_cols<3>)
    const uint32_t tw = (n_ranks + 1) & ~1u;
    const size_t slot_bytes = 10 + 4 * (size_t)tw;
    const uint32_t slots = (uint32_t)std::min<size_t>(kAggMaxSlots, (agg_smem_budget(c) - 8) / slot_bytes - kMaxProbe);
    const size_t smem = (((size_t)slots + kMaxProbe) * slot_bytes + 8 + 15) & ~size_t(15);
    for (uint32_t s = 0; s < n_ranks; ++s)
        if (src_counts[s] >= 0xFFFFFFFFULL) return fail(c, GRMKM_E_UNSUPPORTED, "more than 2^32 partial columns from one source");
    // an owner sees 1/P of the hash space: size the buckets for n_total * P entries over the full range
    const uint64_t per = std::max<uint64_t>(1, slots / 2);
    uint32_t mb = std::min(24u, std::max(6u, ceil_log2((n_total * owners + per - 1) / per)));
    if (const char* e = getenv("GRMKM_MERGE_BITS")) mb = (uint32_t)std::min(24, std::max(6, atoi(e)));      // tests: a merge grid finer than the owners' grid
    if (partial_out) mb = std::max(mb, ob);          // the export cuts the merged chunks on the owners' grid: never coarser than that
    // This owner's slice of the bucket space: the hash range [own_lo, own_hi) of the owners' grid (2^ob buckets), scaled
    // exactly when the merge grid is finer, the enclosing buckets when it is coarser (the sources hold nothing outside
    // the owner's range).
    uint32_t b_lo, b_hi;
    if (mb >= ob) { b_lo = (uint32_t)(own_lo << (mb - ob)); b_hi = (uint32_t)(own_hi << (mb - ob)); }
    else { b_lo = (uint32_t)(own_lo >> (ob - mb)); b_hi = (uint32_t)((own_hi + (1ULL << (ob - mb)) - 1) >> (ob - mb)); }
    const uint32_t nb = b_hi - b_lo, nb1 = nb + 1;
    ENSURE(c, c->scalars, S_COUNT * 8);
    ENSURE(c, c->offsets2, (size_t)(nb + 1) * 8);
    ENSURE(c, c->bbase, (size_t)nb * 8);
    ENSURE(c, c->bcounts, (size_t)nb * 8);
    ENSURE(c, c->refs, (size_t)n_ranks * nb1 * 8 + 16 * 8 * 3);      // bounds + source tables
    uint64_t ucap = std::min<uint64_t>(n_total, 0xFFFFFFFFULL);
    // ordered emission (as in a final one-GPU build): the merge buckets are dealt by ticket and every bucket learns its
    // offset by look-back, so the slice's columns land at their final place and no gather pass follows
    const bool ordered = !partial_out && !getenv("GRMKM_UNORDERED");
    if (ordered) {
        ENSURE(c, c->kmers, ucap * 8);
        ENSURE(c, c->matrix, (size_t)ucap * W_total * 8);
        ENSURE(c, c->apub, (size_t)(nb + 1) * 8);
    } else {
        ENSURE(c, c->ukeys, ucap * 8);
        ENSURE(c, c->uwords, (size_t)ucap * W_total * 8);
    }
    uint64_t* d_scalars = (uint64_t*)c->scalars.p;
    unsigned long long* d_bounds = (unsigned long long*)c->refs.p;
    unsigned long long* d_meta = d_bounds + (size_t)n_ranks * nb1;
    if (c->ev_ok) cudaEventRecord(c->ev[T_START], st);
    CU_TRY(c, cudaMemsetAsync(c->scalars.p, 0, S_COUNT * 8, st));
    if (ordered) CU_TRY(c, cudaMemsetAsync(c->apub.p, 0, (size_t)(nb + 1) * 8, st));
    for (uint32_t s = 0; s < 16; ++s) h_meta[32 + s] = 0;
    memcpy(&h_meta[32], h_width, sizeof h_width);
    CU_TRY(c, cudaMemcpyAsync(d_meta, h_meta.data(), 48 * 8, cudaMemcpyHostToDevice, st));
    const unsigned long long* parts = (const unsigned long long*)dev_parts;
    const uint64_t n_search = (uint64_t)n_ranks * nb1;
    k_merge_bounds<<<(uint32_t)((n_search + 255) / 256), 256, 0, st>>>(parts, n_ranks, nb1, b_lo, mb, d_meta, d_meta + 16,
                                                                      (const uint32_t*)(d_meta + 32), d_bounds);
    L.n++;
    CU_TRY(c, cudaGetLastError());
    if (c->ev_ok) cudaEventRecord(c->ev[T_SCATTER], st);
    ap.bucket_bits = mb; ap.row_bits = 0; ap.n_words = W_total; ap.slots = slots;
    ap.keep_singletons = partial_out ? 1u : c->cfg.keep_singletons; ap.sub_bits = 0; ap.table_u32 = tw;
    ap.partial_out = partial_out ? 1u : 0u;
    ap.out_keys = (unsigned long long*)c->ukeys.p; ap.out_words = (unsigned long long*)c->uwords.p;
    ap.cap = ucap; ap.scalars = (unsigned long long*)d_scalars; ap.parts = parts; ap.bounds = d_bounds;
    ap.bucket_base = (unsigned long long*)c->bbase.p; ap.bucket_count = (unsigned long long*)c->bcounts.p;
    ap.b_begin = b_lo; ap.b_end = b_hi;
    if (ordered) {
        ap.ordered = 1;
        ap.out_keys = (unsigned long long*)c->kmers.p; ap.out_words = (unsigned long long*)c->matrix.p;      // row pitch = ucap
        ap.pub = (unsigned long long*)c->apub.p; ap.ticket = (unsigned int*)((unsigned long long*)c->apub.p + nb);
    }
    CU_TRY(c, cudaFuncSetAttribute(k_aggregate_cols<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_aggregate_cols<3><<<std::max(1u, std::min<uint32_t>(nb, (uint32_t)c->sm_count * kAggCtasPerSm)), kAggThreads, smem, st>>>(ap);
    L.n++;
    CU_TRY(c, cudaGetLastError());
    if (c->ev_ok) cudaEventRecord(c->ev[T_AGG], st);
    uint64_t sc[S_COUNT];
    CU_TRY(c, cudaMemcpyAsync(sc, d_scalars, sizeof sc, cudaMemcpyDeviceToHost, st));
    if (ordered && c->ev_ok) cudaEventRecord(c->ev[T_SORT], st);
    CU_TRY(c, cudaStreamSynchronize(st));
    const uint64_t U = sc[S_U_NEEDED];
    if (partial_out) {
        // the merged partial columns stay as bucket chunks (ukeys / uwords), like the output of a partial build
        ENSURE(c, c->offsets2, (size_t)(nb + 1) * 8);
        k_bucket_offsets<<<1, 1024, 0, st>>>((unsigned long long*)c->bcounts.p, (unsigned long long*)c->offsets2.p, nb,
                                             d_scalars, S_N_SOLID, 1);
        L.n++;
        CU_TRY(c, cudaGetLastError());
        c->merge_h_off.resize(nb + 1);
        CU_TRY(c, cudaMemcpyAsync(c->merge_h_off.data(), c->offsets2.p, (size_t)(nb + 1) * 8, cudaMemcpyDeviceToHost, st));
        if (c->ev_ok) cudaEventRecord(c->ev[T_SORT], st);
        CU_TRY(c, cudaStreamSynchronize(st));
        c->merge_bits = mb; c->merge_cap = ucap;
    } else if (!ordered) {
        ENSURE(c, c->kmers, U * 8);
        ENSURE(c, c->matrix, (size_t)U * W_total * 8);
        k_bucket_offsets<<<1, 1024, 0, st>>>((unsigned long long*)c->bcounts.p, (unsigned long long*)c->offsets2.p, nb,
                                             d_scalars, S_N_SOLID, 1);
        if (U) {
            k_gather_buckets<<<std::max(1u, std::min<uint32_t>(nb, (uint32_t)c->sm_count * 8)), 256, 0, st>>>(
                (const unsigned long long*)c->ukeys.p, (const unsigned long long*)c->uwords.p, ucap,
                (const unsigned long long*)c->bbase.p, (const unsigned long long*)c->offsets2.p, nb, W_total, U,
                (unsigned long long*)c->kmers.p, (unsigned long long*)c->matrix.p, U);
        }
        L.n += 2;
        CU_TRY(c, cudaGetLastError());
        if (c->ev_ok) cudaEventRecord(c->ev[T_SORT], st);
        CU_TRY(c, cudaStreamSynchronize(st));
    }
    c->U = U; c->built = !partial_out;
    c->pitch = ordered ? ucap : U;
    c->stats.n_kmers = U; c->stats.n_distinct = sc[S_N_DISTINCT]; c->stats.n_words = W_total;
    c->stats.n_genomes = total_genomes; c->stats.n_splits += sc[S_N_SPLITS];
    c->stats.n_launches = launches_before + L.n;
    if (c->ev_ok && inside_build) {
        float t = 0.f;                         // the row-block merge of a build counts as its ordering stage
        if (cudaEventElapsedTime(&t, c->ev[T_START], c->ev[T_SORT]) == cudaSuccess) { c->times.sort += t; c->times.total += t; }
        else cudaGetLastError();
    } else if (c->ev_ok) {
        cudaEventElapsedTime(&c->times.scatter, c->ev[T_START], c->ev[T_SCATTER]);
        cudaEventElapsedTime(&c->times.aggregate, c->ev[T_SCATTER], c->ev[T_AGG]);
        cudaEventElapsedTime(&c->times.sort, c->ev[T_AGG], c->ev[T_SORT]);
        cudaEventElapsedTime(&c->times.total, c->ev[T_START], c->ev[T_SORT]);
    }
    return GRMKM_OK;
}


extern "C" {

int grmkm_merge_partials(grmkm_ctx* c, const void* dev_parts, uint32_t n_ranks, uint32_t rank, const uint64_t* src_counts,
                         const uint32_t* src_words, uint32_t total_genomes) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (n_ranks < 1 || n_ranks > 16 || rank >= n_ranks || !src_counts || !src_words)
        return fail(c, GRMKM_E_INVALID, "bad merge arguments");
    // Ownership was dealt on the grid of the partial builds (2^ob buckets, ob = the agreed bucket count capped like
    // build_impl caps it): owner r holds buckets [floor(B r / P), floor(B (r + 1) / P)) of THAT grid.
    if (n_ranks > 1 && !c->cfg.bucket_bits)
        return fail(c, GRMKM_E_INVALID, "grmkm_merge_partials needs the bucket count the partial builds agreed on (grmkm_set_bucket_bits)");
    const uint32_t ob = n_ranks > 1 ? std::min(kUnitMaxBucketBits, c->cfg.bucket_bits) : 0u;
    const uint64_t own_lo = ((1ULL << ob) * rank) / n_ranks, own_hi = ((1ULL << ob) * (rank + 1)) / n_ranks;
    forget_result(c);
    const int r = merge_sources(c, dev_parts, n_ranks, src_counts, src_words, total_genomes, ob, own_lo, own_hi, n_ranks, false, false);
    c->slice = r == GRMKM_OK && n_ranks > 1;
    return r;
}

// ------------------------------------------------------------------------------------------------
// kernels over the finished result (grmkm_result.cuh)
// ------------------------------------------------------------------------------------------------
int grmkm_result_checksum(grmkm_ctx* c, uint64_t out[2]) {
    if (check_ctx(c) || !out) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    out[0] = out[1] = 0;
    if (!c->U) return GRMKM_OK;
    CU_TRY(c, cudaSetDevice(c->device));
    ENSURE(c, c->aux, 16);
    CU_TRY(c, cudaMemsetAsync(c->aux.p, 0, 16, c->stream));
    k_checksum<<<(uint32_t)std::min<uint64_t>((c->U + 255) / 256, (uint64_t)c->sm_count * 8), 256, 0, c->stream>>>(
        (const unsigned long long*)c->kmers.p, (const unsigned long long*)c->matrix.p, c->U, c->pitch, c->W, (unsigned long long*)c->aux.p);
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches++;
    CU_TRY(c, cudaMemcpyAsync(out, c->aux.p, 16, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_sum_rows(grmkm_ctx* c, const uint64_t* row_mask, uint32_t n_mask_words, uint32_t* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    if (cap < c->U) return fail(c, GRMKM_E_CAPACITY, "sum buffer too small");
    if (n_mask_words != c->W || (c->W && !row_mask)) return fail(c, GRMKM_E_INVALID, "the row mask has one word per matrix word row");
    if (c->W > 512) return fail(c, GRMKM_E_UNSUPPORTED, "row masks of more than 512 words");
    if (!c->U) return GRMKM_OK;
    if (!dst) return fail(c, GRMKM_E_INVALID, "null dst");
    CU_TRY(c, cudaSetDevice(c->device));
    const size_t mask_bytes = ((size_t)c->W * 8 + 255) & ~size_t(255);
    ENSURE(c, c->aux, mask_bytes + c->U * 4);
    uint32_t* d_out = (uint32_t*)((uint8_t*)c->aux.p + mask_bytes);
    CU_TRY(c, cudaMemcpyAsync(c->aux.p, row_mask, (size_t)c->W * 8, cudaMemcpyHostToDevice, c->stream));
    k_sum_rows<<<(uint32_t)std::min<uint64_t>((c->U + 255) / 256, (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(
        (const unsigned long long*)c->matrix.p, c->U, c->pitch, c->W, (const unsigned long long*)c->aux.p, d_out);
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches++;
    CU_TRY(c, cudaMemcpyAsync(dst, d_out, c->U * 4, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_gram(grmkm_ctx* c, uint64_t* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build first");
    const uint64_t G = c->G;
    if (cap < G * G) return fail(c, GRMKM_E_CAPACITY, "gram buffer too small");
    if (!G) return GRMKM_OK;
    if (!dst) return fail(c, GRMKM_E_INVALID, "null dst");
    if (!c->U) { memset(dst, 0, G * G * 8); return GRMKM_OK; }
    CU_TRY(c, cudaSetDevice(c->device));
    const uint64_t UW = (c->U + 63) / 64;
    const size_t rows_bytes = (size_t)c->W * 64 * UW * 8;
    ENSURE(c, c->aux, rows_bytes + G * G * 8);
    unsigned long long* d_rows = (unsigned long long*)c->aux.p;
    unsigned long long* d_gram = (unsigned long long*)((uint8_t*)c->aux.p + rows_bytes);
    k_bit_rows<<<(uint32_t)std::min<uint64_t>(((uint64_t)c->W * UW + 7) / 8, (uint64_t)c->sm_count * 32), 256, 0, c->stream>>>(
        (const unsigned long long*)c->matrix.p, c->U, c->pitch, c->W, UW, d_rows);
    k_gram<<<(uint32_t)std::min<uint64_t>(G * (G + 1) / 2, (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(d_rows, UW, (uint32_t)G, d_gram);
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches += 2;
    CU_TRY(c, cudaMemcpyAsync(dst, d_gram, G * G * 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

int grmkm_tsv_pack(grmkm_ctx* c, const uint8_t* body, uint64_t n_rows, uint32_t row_width, uint32_t k, uint32_t n_tsv_cols,
                   uint32_t n_genomes, const uint32_t* sel, uint64_t* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    const uint32_t W = (n_genomes + 63) / 64;
    if (row_width != k + 2 * n_tsv_cols + 1) return fail(c, GRMKM_E_INVALID, "row width is not k + 2 x columns + 1");
    if (cap < n_rows * W) return fail(c, GRMKM_E_CAPACITY, "matrix buffer too small");
    if (n_genomes && !sel) return fail(c, GRMKM_E_INVALID, "null column selection");
    for (uint32_t g = 0; g < n_genomes; ++g) if (sel[g] >= n_tsv_cols) return fail(c, GRMKM_E_INVALID, "column selection out of range");
    if (!n_rows || !W) return GRMKM_OK;
    if (!body || !dst) return fail(c, GRMKM_E_INVALID, "null buffer");
    CU_TRY(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    // staged in chunks of rows: H2D of chunk i + 1 is queued behind the kernel of chunk i on the same stream (the text
    // arrives from pageable memory, so the copy itself is the bound)
    const uint64_t rows_per = std::max<uint64_t>(1, (256ULL << 20) / row_width);
    const size_t sel_bytes = ((size_t)n_genomes * 4 + 255) & ~size_t(255);
    ENSURE(c, c->aux, sel_bytes + 256 + (size_t)n_rows * W * 8);
    ENSURE(c, c->fmt, std::min<uint64_t>(n_rows, rows_per) * row_width);
    uint32_t* d_sel = (uint32_t*)c->aux.p;
    unsigned int* d_bad = (unsigned int*)((uint8_t*)c->aux.p + sel_bytes);
    unsigned long long* d_mat = (unsigned long long*)((uint8_t*)c->aux.p + sel_bytes + 256);
    CU_TRY(c, cudaMemcpyAsync(d_sel, sel, (size_t)n_genomes * 4, cudaMemcpyHostToDevice, st));
    CU_TRY(c, cudaMemsetAsync(d_bad, 0, 4, st));
    for (uint64_t j0 = 0; j0 < n_rows; j0 += rows_per) {
        const uint64_t rows = std::min(rows_per, n_rows - j0);
        CU_TRY(c, cudaMemcpyAsync(c->fmt.p, body + j0 * row_width, rows * row_width, cudaMemcpyHostToDevice, st));
        k_tsv_pack<<<(uint32_t)std::min<uint64_t>((rows + 7) / 8, (uint64_t)c->sm_count * 32), 256, 0, st>>>(
            (const uint8_t*)c->fmt.p, rows, row_width, k, n_genomes, d_sel, j0, n_rows, d_mat, d_bad);
        CU_TRY(c, cudaGetLastError());
        c->stats.n_launches++;
    }
    unsigned int bad = 0;
    CU_TRY(c, cudaMemcpyAsync(dst, d_mat, (size_t)n_rows * W * 8, cudaMemcpyDeviceToHost, st));
    CU_TRY(c, cudaMemcpyAsync(&bad, d_bad, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(c, cudaStreamSynchronize(st));
    if (bad) return fail(c, GRMKM_E_INVALID, "the k-mer matrix is not binary (cells must be 0 or 1)");
    return GRMKM_OK;
}

int grmkm_load_result(grmkm_ctx* c, const uint64_t* kmers, const uint64_t* matrix, uint64_t n_kmers, uint32_t n_genomes) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (n_genomes > kMaxGenomes) return fail(c, GRMKM_E_UNSUPPORTED, "at most 32768 genomes in one context");
    const uint32_t W = (n_genomes + 63) / 64;
    if (n_kmers && (!kmers || (W && !matrix))) return fail(c, GRMKM_E_INVALID, "null kmers or matrix");
    if (n_genomes % 64 && n_kmers) {
        const uint64_t beyond = ~0ULL >> (n_genomes % 64);     // bits of rows n_genomes .. 64 W - 1 in the last word row
        const uint64_t* last = matrix + (uint64_t)(W - 1) * n_kmers;
        for (uint64_t j = 0; j < n_kmers; ++j)
            if (last[j] & beyond) return fail(c, GRMKM_E_INVALID, "the matrix has set bits at rows >= n_genomes");
    }
    CU_TRY(c, cudaSetDevice(c->device));
    if (c->aux_stream) CU_TRY(c, cudaStreamSynchronize(c->aux_stream));
    c->built = false;
    ENSURE(c, c->kmers, n_kmers * 8);
    ENSURE(c, c->matrix, n_kmers * W * 8);
    if (n_kmers) {
        CU_TRY(c, cudaMemcpyAsync(c->kmers.p, kmers, n_kmers * 8, cudaMemcpyHostToDevice, c->stream));
        if (W) CU_TRY(c, cudaMemcpyAsync(c->matrix.p, matrix, n_kmers * W * 8, cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
    }
    c->U = n_kmers; c->W = W; c->G = n_genomes; c->pitch = n_kmers;
    set_result(c, true);
    c->stats.h2d_bytes = n_kmers * (W + 1) * 8;
    return GRMKM_OK;
}

}  // extern "C"

namespace {

double scm_unkey(uint64_t k) {
    const uint64_t b = (k >> 63) ? (k & ~(1ULL << 63)) : ~k;
    double u;
    memcpy(&u, &b, 8);
    return u;
}

// ------------------------------------------------------------------------------------------------
// sharded runs: one rank's slice of the global matrix and the all-gather the ranks talk through
// ------------------------------------------------------------------------------------------------
struct Shard {
    uint32_t rank = 0, n_ranks = 1;
    uint64_t off = 0, total = 0;            // this slice's first global column; U of the whole matrix
    grmkm_exchange_fn fn = nullptr;         // nullptr: the whole matrix on one rank, nothing exchanged
    void* user = nullptr;
    std::vector<uint64_t> offs;             // every rank's first column and offs[n_ranks] = total (from the first exchange)
    bool on() const { return fn != nullptr; }
    uint32_t owner(uint64_t j) const { return (uint32_t)(std::upper_bound(offs.begin(), offs.end(), j) - offs.begin() - 1); }
    bool mine(uint64_t j) const { return j >= offs[rank] && j < offs[rank + 1]; }
    // a global rule (j or total + j) -> the local rule of this slice of U columns (j or U + j)
    uint64_t local_rule(uint64_t r, uint64_t U) const { return r < total ? r - off : U + (r - total - off); }
    uint64_t global_rule(uint64_t r, uint64_t U) const { return r < U ? off + r : total + off + (r - U); }
};

// The Shard of a learner entry point: the plain call (refusal: what it answers for a slice) runs on the whole matrix,
// the sharded call (refusal null) on the slice `in` describes.
int run_shard(grmkm_ctx* c, const grmkm_shard* in, const char* refusal, Shard& s) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (refusal) {
        if (c->built && c->slice) return fail(c, GRMKM_E_UNSUPPORTED, refusal);
        s.total = c->U;
        s.offs = {0, c->U};
        return GRMKM_OK;
    }
    if (!in) return fail(c, GRMKM_E_INVALID, "null shard");
    if (in->struct_size != sizeof(grmkm_shard)) return fail(c, GRMKM_E_INVALID, "shard struct_size is not sizeof(grmkm_shard)");
    if (!in->exchange) return fail(c, GRMKM_E_INVALID, "null shard exchange");
    if (in->n_ranks == 0 || in->rank >= in->n_ranks || in->reserved != 0)
        return fail(c, GRMKM_E_INVALID, "shard rank must be below n_ranks, and reserved 0");
    s.rank = in->rank; s.n_ranks = in->n_ranks;
    s.off = in->col_offset; s.total = in->n_kmers_total;
    s.fn = in->exchange; s.user = in->user;
    return GRMKM_OK;
}

// one all-gather: blk[r] / len[r] = the bytes rank r sent
struct Gathered {
    std::vector<const uint8_t*> blk;
    std::vector<uint64_t> len;
};

int shard_exchange(grmkm_ctx* c, const Shard& s, const void* send, uint64_t n, Gathered& g) {
    const void* recv = nullptr;
    g.len.assign(s.n_ranks, 0);
    if (s.fn(s.user, send, n, &recv, g.len.data()) != 0)
        return fail(c, GRMKM_E_INVALID, "the shard exchange failed on rank " + std::to_string(s.rank));
    if (g.len[s.rank] != n) return fail(c, GRMKM_E_INVALID, "the shard exchange returned a block of another size for this rank");
    g.blk.resize(s.n_ranks);
    uint64_t o = 0;
    for (uint32_t r = 0; r < s.n_ranks; ++r) { g.blk[r] = (const uint8_t*)recv + o; o += g.len[r]; }
    return GRMKM_OK;
}

// The first exchange of a sharded run: every rank's validation status, column range and n_kmers_total.  If any rank
// failed, every rank returns the code of the first failing one, before any device work; ranges that do not tile
// [0, n_kmers_total), or ranks that disagree on n_kmers_total, fail every rank too.  Otherwise s.offs is filled.
int shard_agree(grmkm_ctx* c, Shard& s, int status) {
    if (!s.on()) return status;
    struct Hello { int32_t status; uint32_t pad; uint64_t off, n, total; };
    const Hello mine{status, 0, s.off, c->built ? c->U : 0, s.total};
    const std::string own_err = c->err;
    Gathered g;
    if (int r = shard_exchange(c, s, &mine, sizeof mine, g)) return r;
    s.offs.assign(s.n_ranks + 1, 0);
    uint64_t next = 0;
    bool tiled = true, same_total = true;
    for (uint32_t r = 0; r < s.n_ranks; ++r) {
        if (g.len[r] != sizeof(Hello)) return fail(c, GRMKM_E_INVALID, "rank " + std::to_string(r) + " is not in this run");
        Hello h;
        memcpy(&h, g.blk[r], sizeof h);
        if (h.status) {
            if (r == s.rank) { c->err = own_err; return h.status; }
            return fail(c, h.status, "rank " + std::to_string(r) + " refused the run");
        }
        tiled = tiled && h.off == next;
        same_total = same_total && h.total == s.total;
        s.offs[r] = h.off;
        next = h.off + h.n;
    }
    s.offs[s.n_ranks] = next;
    if (!same_total) return fail(c, GRMKM_E_INVALID, "the ranks were given different n_kmers_total");
    if (!tiled || next != s.total)
        return fail(c, GRMKM_E_INVALID, "the column slices do not tile [0, n_kmers_total) in rank order");
    return GRMKM_OK;
}

// dst[w][i] = the words of local columns idx[i], i < m (< 2^32), packed on the device by k_gather_columns
int pack_columns(grmkm_ctx* c, const uint64_t* idx, uint64_t m, uint64_t* dst) {
    const uint32_t W = c->W;
    if (!m || !W) return GRMKM_OK;
    ENSURE(c, c->shard_idx, m * 8 + m * W * 8);
    unsigned long long* d_idx = (unsigned long long*)c->shard_idx.p;
    CU_TRY(c, cudaMemcpyAsync(d_idx, idx, m * 8, cudaMemcpyHostToDevice, c->stream));
    k_gather_columns<<<(uint32_t)std::min<uint64_t>((m + 7) / 8, (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(
        (const unsigned long long*)c->matrix.p, c->pitch, W, d_idx, (uint32_t)m, d_idx + m);
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches++;
    CU_TRY(c, cudaMemcpyAsync(dst, d_idx + m, m * W * 8, cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

// The matrix a step reads the columns it chose from.  On the whole matrix it is the resident one and global column j is
// its column j.  On a slice it is the compact [W][n] matrix of the n distinct chosen columns, and global column j is its
// position among them.
struct ColumnView {
    const unsigned long long* matrix = nullptr;
    uint64_t U = 0, pitch = 0;
    bool whole = true;
    std::vector<uint64_t> cols;             // a slice's view: the distinct global columns, ascending
    uint64_t col(uint64_t j) const {
        return whole ? j : (uint64_t)(std::lower_bound(cols.begin(), cols.end(), j) - cols.begin());
    }
    // a global rule (j or UG + j) -> the rule of the view (col(j) or U + col(j))
    uint64_t rule(uint64_t r, uint64_t UG) const { return col(r % UG) + (r >= UG ? U : 0); }
};

// cols: the global columns the step needs, the same list on every rank (any order, repeats allowed).  On a slice every
// rank packs the ones it owns (k_gather_columns), one exchange, and every rank assembles the whole in c->shard_cols.
int column_view(grmkm_ctx* c, const Shard& sh, std::vector<uint64_t> cols, ColumnView& v) {
    v.matrix = (const unsigned long long*)c->matrix.p;
    v.whole = !sh.on();
    if (v.whole) {
        v.U = c->U; v.pitch = c->pitch;
        return GRMKM_OK;
    }
    std::sort(cols.begin(), cols.end());
    cols.erase(std::unique(cols.begin(), cols.end()), cols.end());
    v.cols = std::move(cols);
    const uint32_t W = c->W;
    const uint64_t n = v.U = v.pitch = v.cols.size();
    if (!n) return GRMKM_OK;
    std::vector<uint64_t> own, cnt(sh.n_ranks, 0);
    for (uint64_t j : v.cols) {
        const uint32_t o = sh.owner(j);
        ++cnt[o];
        if (o == sh.rank) own.push_back(j - sh.off);
    }
    const uint64_t m = own.size();
    std::vector<uint64_t> packed(m * W);
    if (int r = pack_columns(c, own.data(), m, packed.data())) return r;
    Gathered g;
    if (int r = shard_exchange(c, sh, packed.data(), m * W * 8, g)) return r;
    for (uint32_t r = 0; r < sh.n_ranks; ++r)
        if (g.len[r] != cnt[r] * W * 8) return fail(c, GRMKM_E_INVALID, "rank " + std::to_string(r) + " sent other columns");
    std::vector<uint64_t> h(n * W), at(sh.n_ranks, 0);
    for (uint64_t i = 0; i < n; ++i) {
        const uint32_t o = sh.owner(v.cols[i]);
        const uint64_t k = at[o]++;
        for (uint32_t w = 0; w < W; ++w) memcpy(&h[(uint64_t)w * n + i], g.blk[o] + ((uint64_t)w * cnt[o] + k) * 8, 8);
    }
    ENSURE(c, c->shard_cols, n * W * 8);
    CU_TRY(c, cudaMemcpyAsync(c->shard_cols.p, h.data(), n * W * 8, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    v.matrix = (const unsigned long long*)c->shard_cols.p;
    return GRMKM_OK;
}

// The exchange between the scan and the tie pass: keys[i] = the max of keys[i] over the ranks, the global best.
// Nothing is exchanged on the whole matrix.  other: the error for a rank that sent another number of keys.
int shard_max(grmkm_ctx* c, const Shard& sh, std::vector<uint64_t>& keys, const char* other) {
    if (!sh.on()) return GRMKM_OK;
    Gathered g;
    if (int r = shard_exchange(c, sh, keys.data(), keys.size() * 8, g)) return r;
    for (uint32_t q = 0; q < sh.n_ranks; ++q) {
        if (g.len[q] != keys.size() * 8) return fail(c, GRMKM_E_INVALID, other);
        for (size_t i = 0; i < keys.size(); ++i) {
            uint64_t x;
            memcpy(&x, g.blk[q] + i * 8, 8);
            keys[i] = std::max(keys[i], x);
        }
    }
    return GRMKM_OK;
}

struct TieList { uint64_t n; const uint8_t* p; };       // one rank's tie list: n entries, its payload at p

// The exchange of the tie lists after the tie pass.  A rank sends [count][payload] with a payload of fixed + per x count
// bytes (the caller's, from block[1] on), or the count alone when its list overflowed (over: count > the list's
// capacity).  If any rank's list overflowed, any_over is set and every rank grows its list and redoes the step, so the
// union is never short; else lists holds every rank's list in rank order.  On the whole matrix the one list is this rank's.
int shard_ties(grmkm_ctx* c, const Shard& sh, uint64_t count, bool over, std::vector<uint64_t>& block, uint64_t fixed,
               uint64_t per, std::vector<TieList>& lists, bool& any_over) {
    any_over = over;
    lists.assign(1, TieList{count, (const uint8_t*)(block.data() + 1)});
    if (!sh.on()) return GRMKM_OK;
    block[0] = count;
    Gathered g;
    if (int r = shard_exchange(c, sh, block.data(), 8 + (over ? 0 : fixed + per * count), g)) return r;
    lists.clear();
    for (uint32_t q = 0; q < sh.n_ranks; ++q) {
        uint64_t n = 0;
        if (g.len[q] < 8) return fail(c, GRMKM_E_INVALID, "a rank sent no tie list");
        memcpy(&n, g.blk[q], 8);
        if (g.len[q] == 8 && n) { any_over = true; continue; }         // an overflow: the count only
        if (g.len[q] != 8 + fixed + per * n) return fail(c, GRMKM_E_INVALID, "a rank sent a malformed tie list");
        lists.push_back(TieList{n, g.blk[q] + 8});
    }
    return GRMKM_OK;
}

// fits or nodes per chunk: as many as share one CTA's shared memory at per_item bytes each, small enough for two CTAs
// per SM
uint32_t chunk_size(const grmkm_ctx* c, size_t per_item) {
    const size_t smem_cap = (c->smem_optin ? c->smem_optin : 227 * 1024) - 1024;
    return (uint32_t)std::max<size_t>(1, std::min<size_t>(smem_cap / 2, 64 * 1024) / per_item);
}

// What every learner run checks first: a result, at most 2^31 - 1 k-mers where the learner indexes them with 32 bits
// (limit: how it says so; null where it does not), and the blacklist.
int check_run(grmkm_ctx* c, const Shard& sh, const char* limit, const uint64_t* blacklist, uint64_t n_blacklist) {
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build or grmkm_load_result first");
    if (limit && sh.total >= (1ULL << 31))
        return fail(c, GRMKM_E_UNSUPPORTED, std::string(limit) + " with 32 bits: at most 2^31 - 1 k-mers");
    if (n_blacklist && !blacklist) return fail(c, GRMKM_E_INVALID, "null blacklist");
    for (uint64_t i = 0; i < n_blacklist; ++i)
        if (blacklist[i] >= 2 * sh.total) return fail(c, GRMKM_E_INVALID, "blacklisted rule index >= 2 x n_kmers");
    return GRMKM_OK;
}

// a job's example masks: not null, no bits at rows >= n_genomes, no example both positive and negative (at: the job)
int check_examples(grmkm_ctx* c, const uint64_t* pos, const uint64_t* neg, const std::string& at) {
    const uint32_t W = c->W;
    if (!W) return GRMKM_OK;
    for (const auto& [m, what] : {std::pair{pos, "positive"}, std::pair{neg, "negative"}}) {
        if (!m) return fail(c, GRMKM_E_INVALID, std::string("null ") + what + " mask");
        if (c->G % 64 && (m[W - 1] & (~0ULL >> (c->G % 64))))
            return fail(c, GRMKM_E_INVALID, std::string("the ") + what + " mask has bits at rows >= n_genomes");
    }
    for (uint32_t w = 0; w < W; ++w)
        if (pos[w] & neg[w]) return fail(c, GRMKM_E_INVALID, "positive and negative examples overlap" + at);
    return GRMKM_OK;
}

// SCM passes over this rank's columns: bit 0 the scan, bit 1 the tie pass (the same grid in both)
enum { SCM_SCAN = 1, SCM_TIES = 2 };

template <bool CACHED>
int scm_launch_chunk(grmkm_ctx* c, int passes, const ScmFitArg* d_args, uint32_t n, const uint32_t* d_bl,
                     const unsigned long long* d_masks, unsigned long long* d_best, unsigned long long* d_tile,
                     unsigned long long* d_list, unsigned long long* d_count, uint64_t cap) {
    if (c->U == 0) return GRMKM_OK;         // a rank without columns (sharded runs): a zero-size grid is a launch error
    const size_t smem = scm_smem_bytes(n, c->W);
    CU_TRY(c, cudaFuncSetAttribute(k_scm_scan<CACHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU_TRY(c, cudaFuncSetAttribute(k_scm_ties<CACHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CU_TRY(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_scm_scan<CACHED>, kScmThreads, smem));
    const uint64_t n_tiles = (c->U + kScmThreads - 1) / kScmThreads;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(n_tiles, (uint64_t)c->sm_count * std::max(1, occ));
    const unsigned long long* m = (const unsigned long long*)c->matrix.p;
    if (passes & SCM_SCAN) {
        k_scm_scan<CACHED><<<grid, kScmThreads, smem, c->stream>>>(m, c->U, c->pitch, c->W, d_bl, d_args, n, d_masks, d_best, d_tile);
        c->stats.n_launches++;
    }
    if (passes & SCM_TIES) {
        k_scm_ties<CACHED><<<grid, kScmThreads, smem, c->stream>>>(m, c->U, c->pitch, c->W, d_bl, d_args, n, d_masks, d_best, d_tile,
                                                                   d_list, d_count, cap);
        c->stats.n_launches++;
    }
    CU_TRY(c, cudaGetLastError());
    return GRMKM_OK;
}

int scm_validate(grmkm_ctx* c, uint32_t n_fits, const grmkm_scm_job* jobs, const uint64_t* blacklist, uint64_t n_blacklist,
                 const Shard& sh) {
    if (int r = check_run(c, sh, "the SCM indexes rules", blacklist, n_blacklist)) return r;
    if (n_fits && !jobs) return fail(c, GRMKM_E_INVALID, "null jobs");
    for (uint32_t f = 0; f < n_fits; ++f) {
        const grmkm_scm_job& j = jobs[f];
        const std::string at = " (fit " + std::to_string(f) + ")";
        if (j.struct_size != sizeof(grmkm_scm_job)) return fail(c, GRMKM_E_INVALID, "job struct_size is not sizeof(grmkm_scm_job)" + at);
        if (j.model_type > GRMKM_SCM_DISJUNCTION) return fail(c, GRMKM_E_INVALID, "unknown model type" + at);
        if (j.max_rules == 0) return fail(c, GRMKM_E_INVALID, "max_rules must be at least 1" + at);
        if (j.tiebreak > 1) return fail(c, GRMKM_E_INVALID, "tiebreak must be 0 or 1" + at);
        if (!(j.p >= 0.0) || j.p > 1.7976931348623157e308) return fail(c, GRMKM_E_INVALID, "p must be finite and >= 0" + at);
        if (int r = check_examples(c, j.pos, j.neg, at)) return r;
    }
    return GRMKM_OK;
}

// The greedy loop of a batch of fits on this rank's columns; sh: the whole matrix (no exchange) or one slice of it.
// Sharded, each step is: scan -> exchange the best keys -> tie pass and statistics against the global keys -> exchange
// the tie lists -> the same host selection on every rank -> exchange the chosen columns -> update the masks.
int scm_run(grmkm_ctx* c, uint32_t n_fits, const grmkm_scm_job* jobs, const uint64_t* blacklist, uint64_t n_blacklist,
            const grmkm_shard* shard, const char* refusal) {
    Shard sh;
    if (int r = run_shard(c, shard, refusal, sh)) return r;
    if (int r = shard_agree(c, sh, scm_validate(c, n_fits, jobs, blacklist, n_blacklist, sh))) return r;
    const uint64_t U = c->U, UG = sh.total;
    const uint32_t W = c->W;
    const bool sharded = sh.on();

    NvtxRange nv("grmkm_scm_run");
    c->scm_steps.assign(n_fits, {});
    c->scm_equiv.assign(n_fits, {});
    std::vector<uint32_t> n_pos(n_fits), n_neg(n_fits), n_rules(n_fits, 0);
    std::vector<char> done(n_fits, 0);
    std::vector<uint64_t> h_masks((size_t)n_fits * 4 * W);
    for (uint32_t f = 0; f < n_fits; ++f) {
        const bool swap = jobs[f].model_type == GRMKM_SCM_DISJUNCTION;
        const uint64_t* P0 = swap ? jobs[f].neg : jobs[f].pos;
        const uint64_t* N0 = swap ? jobs[f].pos : jobs[f].neg;
        uint32_t np = 0, nn = 0;
        for (uint32_t w = 0; w < W; ++w) {
            uint64_t* m = h_masks.data() + (size_t)f * 4 * W;
            m[w] = m[2 * W + w] = P0[w];
            m[W + w] = m[3 * W + w] = N0[w];
            np += (uint32_t)__builtin_popcountll(P0[w]);
            nn += (uint32_t)__builtin_popcountll(N0[w]);
        }
        n_pos[f] = np; n_neg[f] = nn;
        done[f] = nn == 0 || UG == 0;         // nothing to cover, or no rule at all
    }
    if (std::find(done.begin(), done.end(), 0) == done.end()) return GRMKM_OK;

    CU_TRY(c, cudaSetDevice(c->device));
    const uint32_t chunk = chunk_size(c, scm_smem_bytes(1, W));
    const uint64_t bl_words = (2 * U + 31) / 32;
    const uint64_t max_grid = (uint64_t)c->sm_count * 8;
    // sharded, the tie pass runs after the exchange of the keys: every chunk keeps its per-CTA bests until then
    const uint64_t tile_fits = sharded ? n_fits : chunk;
    auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t o_masks = 0, o_best = o_masks + al(h_masks.size() * 8), o_args = o_best + al((size_t)n_fits * 8),
                 o_bl = o_args + al((size_t)n_fits * sizeof(ScmFitArg)), o_tile = o_bl + al(bl_words * 4),
                 o_sel = o_tile + al((size_t)tile_fits * max_grid * 8), o_count = o_sel + al((size_t)n_fits * 8),
                 total = o_count + 256;
    ENSURE(c, c->scm, total);
    uint8_t* base = (uint8_t*)c->scm.p;
    unsigned long long* d_masks = (unsigned long long*)(base + o_masks);
    unsigned long long* d_best = (unsigned long long*)(base + o_best);
    ScmFitArg* d_args = (ScmFitArg*)(base + o_args);
    uint32_t* d_bl = (uint32_t*)(base + o_bl);
    unsigned long long* d_tile = (unsigned long long*)(base + o_tile);
    unsigned long long* d_sel = (unsigned long long*)(base + o_sel);
    unsigned long long* d_count = (unsigned long long*)(base + o_count);
    std::vector<uint32_t> h_bl(bl_words, 0);
    for (uint64_t i = 0; i < n_blacklist; ++i) {
        const uint64_t b = blacklist[i];
        if (!sh.mine(b % UG)) continue;
        const uint64_t r = sh.local_rule(b, U);
        h_bl[r >> 5] |= 1u << (r & 31);
    }
    CU_TRY(c, cudaMemcpyAsync(d_masks, h_masks.data(), h_masks.size() * 8, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(c, cudaMemcpyAsync(d_bl, h_bl.data(), bl_words * 4, cudaMemcpyHostToDevice, c->stream));

    uint64_t cap = std::max<uint64_t>(1024, c->scm_list.cap / 20);      // tie list entries (8 bytes + 3 x 4 bytes of statistics)
    std::vector<ScmFitArg> args;
    std::vector<uint64_t> h_list, h_best(n_fits), sel, keys, block, cols;
    std::vector<uint32_t> h_stats;
    std::vector<size_t> order;
    std::vector<TieList> lists;
    auto launch = [&](int passes) -> int {
        for (size_t a0 = 0; a0 < args.size(); a0 += chunk) {
            const uint32_t n = (uint32_t)std::min<size_t>(chunk, args.size() - a0);
            unsigned long long* tile = d_tile + (sharded ? a0 * max_grid : 0);
            unsigned long long* d_list = (unsigned long long*)c->scm_list.p;
            const int r = W <= kScmCachedWords
                              ? scm_launch_chunk<true>(c, passes, d_args + a0, n, d_bl, d_masks, d_best, tile, d_list, d_count, cap)
                              : scm_launch_chunk<false>(c, passes, d_args + a0, n, d_bl, d_masks, d_best, tile, d_list, d_count, cap);
            if (r) return r;
        }
        return GRMKM_OK;
    };
    for (;;) {
        args.clear();
        for (uint32_t f = 0; f < n_fits; ++f)
            if (!done[f]) args.push_back(ScmFitArg{jobs[f].p, f, n_pos[f], n_neg[f], 0});
        if (args.empty()) break;
        ENSURE(c, c->scm_list, cap * 20);
        unsigned long long* d_list = (unsigned long long*)c->scm_list.p;
        uint32_t* d_stats = (uint32_t*)(d_list + cap);
        CU_TRY(c, cudaMemcpyAsync(d_args, args.data(), args.size() * sizeof(ScmFitArg), cudaMemcpyHostToDevice, c->stream));
        CU_TRY(c, cudaMemsetAsync(d_best, 0, (size_t)n_fits * 8, c->stream));
        CU_TRY(c, cudaMemsetAsync(d_count, 0, 8, c->stream));
        if (!sharded) {
            if (int r = launch(SCM_SCAN | SCM_TIES)) return r;
        } else {
            // exchange 1: the best key of every pending fit, the max over the ranks is the global u*
            if (int r = launch(SCM_SCAN)) return r;
            CU_TRY(c, cudaMemcpyAsync(h_best.data(), d_best, (size_t)n_fits * 8, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(c, cudaStreamSynchronize(c->stream));
            keys.resize(args.size());
            for (size_t a = 0; a < args.size(); ++a) keys[a] = h_best[args[a].fit];
            if (int r = shard_max(c, sh, keys, "a rank sent keys of other fits")) return r;
            for (size_t a = 0; a < args.size(); ++a) h_best[args[a].fit] = keys[a];
            CU_TRY(c, cudaMemcpyAsync(d_best, h_best.data(), (size_t)n_fits * 8, cudaMemcpyHostToDevice, c->stream));
            if (int r = launch(SCM_TIES)) return r;
        }
        uint64_t count = 0;
        CU_TRY(c, cudaMemcpyAsync(&count, d_count, 8, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        const bool over = count > cap;
        if (over && !sharded) {         // the tie list overflowed: grow it and redo the step (nothing was updated)
            cap = count + count / 4;
            continue;
        }
        const uint64_t n_local = over ? 0 : count;
        if (n_local) {
            k_scm_gather<<<(uint32_t)std::min<uint64_t>((count + 255) / 256, (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(
                (const unsigned long long*)c->matrix.p, U, c->pitch, W, d_masks, d_list, count, d_stats);
            CU_TRY(c, cudaGetLastError());
            c->stats.n_launches++;
        }
        h_list.resize(n_local); h_stats.resize(n_local * 3);
        CU_TRY(c, cudaMemcpyAsync(h_list.data(), d_list, n_local * 8, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaMemcpyAsync(h_stats.data(), d_stats, n_local * 12, cudaMemcpyDeviceToHost, c->stream));
        if (!sharded) CU_TRY(c, cudaMemcpyAsync(h_best.data(), d_best, (size_t)n_fits * 8, cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(c, cudaStreamSynchronize(c->stream));
        if (sharded) {
            // exchange 2: the tie lists with global rules, then their statistics (20 bytes per entry)
            block.assign(1 + n_local + (n_local * 3 + 1) / 2, 0);
            for (uint64_t i = 0; i < n_local; ++i)
                block[1 + i] = (h_list[i] & ~0xffffffffULL) | sh.global_rule(h_list[i] & 0xffffffffULL, U);
            if (n_local) memcpy(block.data() + 1 + n_local, h_stats.data(), n_local * 12);
            bool any_over = false;
            if (int r = shard_ties(c, sh, count, over, block, 0, 20, lists, any_over)) return r;
            if (over) cap = count + count / 4;
            if (any_over) continue;
            h_list.clear(); h_stats.clear();
            for (const TieList& l : lists) {
                const size_t l0 = h_list.size();
                h_list.resize(l0 + l.n); h_stats.resize((l0 + l.n) * 3);
                memcpy(h_list.data() + l0, l.p, l.n * 8);
                memcpy(h_stats.data() + l0 * 3, l.p + l.n * 8, l.n * 12);
            }
            count = h_list.size();
        }
        // the list comes in the order of the atomics: sort it by (fit, rule)
        order.resize(count);
        for (size_t i = 0; i < count; ++i) order[i] = i;
        std::sort(order.begin(), order.end(), [&](size_t a, size_t b) { return h_list[a] < h_list[b]; });
        sel.clear();
        size_t i = 0;
        for (const ScmFitArg& a : args) {
            const uint32_t f = a.fit;
            while (i < count && (h_list[order[i]] >> 32) < f) ++i;
            size_t end = i;
            while (end < count && (h_list[order[end]] >> 32) == f) ++end;
            if (end == i) { done[f] = 1; continue; }        // no rule changes anything at u*, or every rule is blacklisted
            uint32_t min_risk = UINT32_MAX;
            if (jobs[f].tiebreak)
                for (size_t t = i; t < end; ++t) min_risk = std::min(min_risk, h_stats[3 * order[t] + 2]);
            std::vector<uint64_t>& eq = c->scm_equiv[f];
            grmkm_scm_step st{};
            st.utility = scm_unkey(h_best[f]);
            st.equiv_offset = eq.size();
            for (size_t t = i; t < end; ++t) {
                const size_t o = order[t];
                if (jobs[f].tiebreak && h_stats[3 * o + 2] != min_risk) continue;
                if (eq.size() == st.equiv_offset) {
                    st.rule = h_list[o] & 0xffffffffULL;
                    st.positive_errors = h_stats[3 * o];
                    st.negative_covers = h_stats[3 * o + 1];
                }
                eq.push_back(h_list[o] & 0xffffffffULL);
            }
            st.equiv_count = eq.size() - st.equiv_offset;
            c->scm_steps[f].push_back(st);
            n_pos[f] -= st.positive_errors;
            n_neg[f] -= st.negative_covers;
            if (n_neg[f] == 0 || ++n_rules[f] == jobs[f].max_rules) done[f] = 1;
            sel.push_back(((uint64_t)f << 32) | st.rule);
            i = end;
        }
        if (!sel.empty()) {
            // exchange 3 on a slice: the chosen columns from their owners; the update runs on their compact matrix
            cols.clear();
            for (uint64_t e : sel) cols.push_back((e & 0xffffffffULL) % UG);
            ColumnView v;
            if (int r = column_view(c, sh, cols, v)) return r;
            for (uint64_t& e : sel) e = (e & ~0xffffffffULL) | v.rule(e & 0xffffffffULL, UG);
            CU_TRY(c, cudaMemcpyAsync(d_sel, sel.data(), sel.size() * 8, cudaMemcpyHostToDevice, c->stream));
            const uint64_t nw = (uint64_t)sel.size() * W;
            k_scm_update<<<(uint32_t)std::min<uint64_t>((nw + 255) / 256, (uint64_t)c->sm_count * 8), 256, 0, c->stream>>>(
                v.matrix, v.U, v.pitch, W, d_sel, (uint32_t)sel.size(), d_masks);
            CU_TRY(c, cudaGetLastError());
            c->stats.n_launches++;
        }
    }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

// one fit's steps or one tree's nodes and their equivalent rules, copied to the caller's buffers (n, n_equivalent: how
// many there are, whether they fit or not)
template <class T>
int copy_result(grmkm_ctx* c, const std::vector<T>& s, const std::vector<uint64_t>& e, T* dst, uint64_t cap, uint64_t* n,
                uint64_t* equivalent, uint64_t equiv_cap, uint64_t* n_equivalent, const char* too_small) {
    if (n) *n = s.size();
    if (n_equivalent) *n_equivalent = e.size();
    if ((!dst && !s.empty()) || cap < s.size() || (!equivalent && !e.empty()) || equiv_cap < e.size())
        return fail(c, GRMKM_E_CAPACITY, too_small);
    if (!s.empty()) memcpy(dst, s.data(), s.size() * sizeof(T));
    if (!e.empty()) memcpy(equivalent, e.data(), e.size() * 8);
    return GRMKM_OK;
}

}  // namespace

extern "C" {

int grmkm_scm_run(grmkm_ctx* c, uint32_t n_fits, const grmkm_scm_job* jobs, const uint64_t* blacklist, uint64_t n_blacklist) {
    return scm_run(c, n_fits, jobs, blacklist, n_blacklist, nullptr,
                   "the result is one owner's slice of a multi-GPU build: its best rule is not the answer");
}

int grmkm_scm_run_sharded(grmkm_ctx* c, uint32_t n_fits, const grmkm_scm_job* jobs, const uint64_t* blacklist,
                          uint64_t n_blacklist, const grmkm_shard* shard) {
    return scm_run(c, n_fits, jobs, blacklist, n_blacklist, shard, nullptr);
}

int grmkm_scm_result(grmkm_ctx* c, uint32_t fit, grmkm_scm_step* steps, uint64_t steps_cap, uint64_t* n_steps,
                     uint64_t* equivalent, uint64_t equiv_cap, uint64_t* n_equivalent) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (fit >= c->scm_steps.size()) return fail(c, GRMKM_E_INVALID, "no such fit in the last grmkm_scm_run");
    return copy_result(c, c->scm_steps[fit], c->scm_equiv[fit], steps, steps_cap, n_steps, equivalent, equiv_cap, n_equivalent,
                       "scm result buffers too small");
}

}  // extern "C"

namespace {

// the largest dynamic shared memory any chunk of this run asks for, set once per run
template <bool CACHED>
int cart_allow_smem(grmkm_ctx* c, size_t smem) {
    CU_TRY(c, cudaFuncSetAttribute(k_cart_scan<CACHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU_TRY(c, cudaFuncSetAttribute(k_cart_ties<CACHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CU_TRY(c, cudaFuncSetAttribute(k_cart_ties<CACHED, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return GRMKM_OK;
}

// the scan (passes bit 0) and both tie passes (bit 1) of one chunk of open nodes; CTA b covers the tiles
// [b tpc, (b + 1) tpc).  A pattern matrix (c->pat_mult_on) counts its tie totals in k-mers (k_cart_ties<., true>).  occ: resident CTAs per SM by chunk size, filled on first use (a run sees few sizes: full chunks
// and the tails of its levels)
template <bool CACHED>
int cart_launch_chunk(grmkm_ctx* c, int passes, const CartNodeArg* d_args, uint32_t n, const uint32_t* d_bl,
                      const unsigned long long* d_masks, unsigned long long* d_best, unsigned long long* d_tile, uint32_t* d_tcnt,
                      unsigned long long* d_total, unsigned long long* d_list, unsigned long long* d_count, uint64_t cap,
                      uint64_t max_grid, std::map<uint32_t, int>& occ_of) {
    if (c->U == 0) return GRMKM_OK;         // a rank without columns (sharded runs): a zero-size grid is a launch error
    const size_t smem = cart_smem_bytes(n, c->W);
    auto it = occ_of.find(n);
    if (it == occ_of.end()) {
        int occ = 0;
        CU_TRY(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_cart_scan<CACHED>, kScmThreads, smem));
        it = occ_of.emplace(n, occ).first;
    }
    const int occ = it->second;
    const uint64_t n_tiles = (c->U + kScmThreads - 1) / kScmThreads;
    const uint64_t grid0 = std::min<uint64_t>({n_tiles, (uint64_t)c->sm_count * std::max(1, occ), max_grid});
    const uint64_t tpc = (n_tiles + grid0 - 1) / grid0;
    const uint32_t grid = (uint32_t)((n_tiles + tpc - 1) / tpc);
    const unsigned long long* m = (const unsigned long long*)c->matrix.p;
    if (passes & SCM_SCAN) {
        k_cart_scan<CACHED><<<grid, kScmThreads, smem, c->stream>>>(m, c->U, c->pitch, c->W, d_bl, d_args, n, d_masks, tpc, d_best, d_tile);
        c->stats.n_launches++;
    }
    if (passes & SCM_TIES) {
        for (int append = 0; append < 2; ++append) {
            if (c->pat_mult_on)
                k_cart_ties<CACHED, true><<<grid, kScmThreads, smem, c->stream>>>(
                    m, c->U, c->pitch, c->W, d_bl, d_args, n, d_masks, tpc, d_best, d_tile, d_tcnt, d_total, append, d_list,
                    d_count, cap, (const uint32_t*)c->pat_mult.p);
            else
                k_cart_ties<CACHED><<<grid, kScmThreads, smem, c->stream>>>(m, c->U, c->pitch, c->W, d_bl, d_args, n, d_masks, tpc, d_best,
                                                                            d_tile, d_tcnt, d_total, append, d_list, d_count, cap);
        }
        c->stats.n_launches += 2;
    }
    CU_TRY(c, cudaGetLastError());
    return GRMKM_OK;
}

int cart_validate(grmkm_ctx* c, uint32_t n_trees, const grmkm_cart_job* jobs, const uint64_t* blacklist, uint64_t n_blacklist,
                  const Shard& sh) {
    if (int r = check_run(c, sh, "CART indexes k-mers", blacklist, n_blacklist)) return r;
    if (n_trees && !jobs) return fail(c, GRMKM_E_INVALID, "null jobs");
    for (uint32_t t = 0; t < n_trees; ++t) {
        const grmkm_cart_job& j = jobs[t];
        const std::string at = " (tree " + std::to_string(t) + ")";
        if (j.struct_size != sizeof(grmkm_cart_job)) return fail(c, GRMKM_E_INVALID, "job struct_size is not sizeof(grmkm_cart_job)" + at);
        if (j.reserved != 0) return fail(c, GRMKM_E_INVALID, "reserved must be 0" + at);
        if (j.max_depth == 0) return fail(c, GRMKM_E_INVALID, "max_depth must be at least 1" + at);
        if (j.min_samples_split < 2) return fail(c, GRMKM_E_INVALID, "min_samples_split must be at least 2" + at);
        if (!(j.w_neg > 0.0 && j.w_neg <= 1e100) || !(j.w_pos > 0.0 && j.w_pos <= 1e100))
            return fail(c, GRMKM_E_INVALID, "class importances must be finite, > 0 and <= 1e100" + at);
        if (int r = check_examples(c, j.pos, j.neg, at)) return r;
    }
    return GRMKM_OK;
}

// The level loop of a batch of trees on this rank's columns; sh: the whole matrix (no exchange) or one slice of it.
// Sharded, each level is: scan -> exchange the best keys -> both tie passes against the global keys -> exchange the
// tie totals and lists -> the same host selection on every rank -> exchange the split columns -> gather and split.
int cart_run(grmkm_ctx* c, uint32_t n_trees, const grmkm_cart_job* jobs, const uint64_t* blacklist, uint64_t n_blacklist,
             const grmkm_shard* shard, const char* refusal) {
    Shard sh;
    if (int r = run_shard(c, shard, refusal, sh)) return r;
    if (int r = shard_agree(c, sh, cart_validate(c, n_trees, jobs, blacklist, n_blacklist, sh))) return r;
    const uint64_t U = c->U, UG = sh.total;
    const uint32_t W = c->W;
    const bool sharded = sh.on();

    NvtxRange nv("grmkm_cart_run");
    c->cart_nodes.assign(n_trees, {});
    c->cart_equiv.assign(n_trees, {});
    struct Open { uint32_t tree, node; };
    std::vector<Open> open, next;
    auto add_node = [&](uint32_t t, uint32_t depth, uint32_t a, uint32_t b) -> uint32_t {
        grmkm_cart_node nd{};
        nd.rule = UINT64_MAX;
        nd.depth = depth; nd.n_pos = a; nd.n_neg = b;
        nd.present_child = nd.absent_child = UINT32_MAX;
        nd.prediction = jobs[t].w_pos * (double)a > jobs[t].w_neg * (double)b;
        c->cart_nodes[t].push_back(nd);
        return (uint32_t)(c->cart_nodes[t].size() - 1);
    };
    // a node is scanned unless a stop rule makes it a leaf first (T empty is only known after the scan)
    auto opens = [&](uint32_t t, uint32_t depth, uint32_t a, uint32_t b) {
        return UG > 0 && depth < jobs[t].max_depth && (uint64_t)a + b >= jobs[t].min_samples_split && a > 0 && b > 0;
    };
    std::vector<uint64_t> h_masks;
    for (uint32_t t = 0; t < n_trees; ++t) {
        uint32_t a = 0, b = 0;
        for (uint32_t w = 0; w < W; ++w) {
            a += (uint32_t)__builtin_popcountll(jobs[t].pos[w]);
            b += (uint32_t)__builtin_popcountll(jobs[t].neg[w]);
        }
        const uint32_t root = add_node(t, 0, a, b);
        if (opens(t, 0, a, b)) {
            open.push_back({t, root});
            h_masks.insert(h_masks.end(), jobs[t].pos, jobs[t].pos + W);
            h_masks.insert(h_masks.end(), jobs[t].neg, jobs[t].neg + W);
        }
    }
    if (open.empty()) return GRMKM_OK;

    CU_TRY(c, cudaSetDevice(c->device));
    const uint32_t chunk = chunk_size(c, cart_smem_bytes(1, W));
    const uint64_t max_grid = (uint64_t)c->sm_count * 8;
    const uint64_t bl_words = (U + 31) / 32;
    std::vector<uint32_t> h_bl(bl_words, 0);
    for (uint64_t i = 0; i < n_blacklist; ++i) {
        const uint64_t j = blacklist[i] % UG;
        if (!sh.mine(j)) continue;
        h_bl[(j - sh.off) >> 5] |= 1u << ((j - sh.off) & 31);
    }
    ENSURE(c, c->cart_bl, bl_words * 4);
    ENSURE(c, c->cart_masks[0], h_masks.size() * 8);
    CU_TRY(c, cudaMemcpyAsync(c->cart_bl.p, h_bl.data(), bl_words * 4, cudaMemcpyHostToDevice, c->stream));
    CU_TRY(c, cudaMemcpyAsync(c->cart_masks[0].p, h_masks.data(), h_masks.size() * 8, cudaMemcpyHostToDevice, c->stream));
    int cur = 0;
    {
        const int r = W <= kScmCachedWords ? cart_allow_smem<true>(c, cart_smem_bytes(chunk, W))
                                           : cart_allow_smem<false>(c, cart_smem_bytes(chunk, W));
        if (r) return r;
    }
    std::map<uint32_t, int> occ_of;

    uint64_t cap = std::max<uint64_t>(1024, c->cart_list.cap / 8);      // tie list entries
    std::vector<CartNodeArg> args;
    std::vector<CartSplit> splits;
    std::vector<uint64_t> h_best, h_total, h_list, block, cols;
    std::vector<uint32_t> h_stats;
    std::vector<TieList> lists;
    auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
    while (!open.empty()) {
        const uint32_t n_open = (uint32_t)open.size();
        // the widest chunk of this level; sharded, the tie passes run after the exchange of the keys, so every chunk
        // keeps its per-CTA bests until then
        const uint32_t cw = std::min(chunk, n_open), tile_nodes = sharded ? n_open : cw;
        args.resize(n_open);
        for (uint32_t i = 0; i < n_open; ++i) {
            const grmkm_cart_job& j = jobs[open[i].tree];
            const grmkm_cart_node& nd = c->cart_nodes[open[i].tree][open[i].node];
            args[i] = CartNodeArg{j.w_pos, j.w_neg, std::max<uint64_t>(1, j.equiv_cap), i, nd.n_pos, nd.n_neg, 0};
        }
        const size_t o_args = 0, o_best = o_args + al((size_t)n_open * sizeof(CartNodeArg)), o_total = o_best + al((size_t)n_open * 8),
                     o_tile = o_total + al((size_t)n_open * 8), o_tcnt = o_tile + al((size_t)tile_nodes * max_grid * 8),
                     o_split = o_tcnt + al((size_t)cw * max_grid * 4), o_stats = o_split + al((size_t)n_open * sizeof(CartSplit)),
                     o_count = o_stats + al((size_t)n_open * 8), total = o_count + 256;
        ENSURE(c, c->cart, total);
        uint8_t* base = (uint8_t*)c->cart.p;
        CartNodeArg* d_args = (CartNodeArg*)(base + o_args);
        unsigned long long* d_best = (unsigned long long*)(base + o_best);
        unsigned long long* d_total = (unsigned long long*)(base + o_total);
        unsigned long long* d_tile = (unsigned long long*)(base + o_tile);
        uint32_t* d_tcnt = (uint32_t*)(base + o_tcnt);
        CartSplit* d_split = (CartSplit*)(base + o_split);
        uint32_t* d_stats = (uint32_t*)(base + o_stats);
        unsigned long long* d_count = (unsigned long long*)(base + o_count);
        const unsigned long long* d_masks = (const unsigned long long*)c->cart_masks[cur].p;
        CU_TRY(c, cudaMemcpyAsync(d_args, args.data(), (size_t)n_open * sizeof(CartNodeArg), cudaMemcpyHostToDevice, c->stream));
        auto launch = [&](int passes) -> int {
            for (uint32_t a0 = 0; a0 < n_open; a0 += chunk) {
                const uint32_t n = std::min(chunk, n_open - a0);
                unsigned long long* tile = d_tile + (sharded ? (uint64_t)a0 * max_grid : 0);
                unsigned long long* d_list = (unsigned long long*)c->cart_list.p;
                const int r = W <= kScmCachedWords
                                  ? cart_launch_chunk<true>(c, passes, d_args + a0, n, (const uint32_t*)c->cart_bl.p, d_masks, d_best,
                                                            tile, d_tcnt, d_total, d_list, d_count, cap, max_grid, occ_of)
                                  : cart_launch_chunk<false>(c, passes, d_args + a0, n, (const uint32_t*)c->cart_bl.p, d_masks, d_best,
                                                             tile, d_tcnt, d_total, d_list, d_count, cap, max_grid, occ_of);
                if (r) return r;
            }
            return GRMKM_OK;
        };
        uint64_t count = 0;
        for (;;) {
            ENSURE(c, c->cart_list, cap * 8);
            CU_TRY(c, cudaMemsetAsync(d_best, 0, (size_t)n_open * 8, c->stream));
            CU_TRY(c, cudaMemsetAsync(d_total, 0, (size_t)n_open * 8, c->stream));
            CU_TRY(c, cudaMemsetAsync(d_count, 0, 8, c->stream));
            if (!sharded) {
                if (int r = launch(SCM_SCAN | SCM_TIES)) return r;
            } else {
                // exchange 1: every open node's best key, the max over the ranks is the global one
                if (int r = launch(SCM_SCAN)) return r;
                h_best.resize(n_open);
                CU_TRY(c, cudaMemcpyAsync(h_best.data(), d_best, (size_t)n_open * 8, cudaMemcpyDeviceToHost, c->stream));
                CU_TRY(c, cudaStreamSynchronize(c->stream));
                if (int r = shard_max(c, sh, h_best, "a rank sent keys of other nodes")) return r;
                CU_TRY(c, cudaMemcpyAsync(d_best, h_best.data(), (size_t)n_open * 8, cudaMemcpyHostToDevice, c->stream));
                if (int r = launch(SCM_TIES)) return r;
            }
            CU_TRY(c, cudaMemcpyAsync(&count, d_count, 8, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(c, cudaStreamSynchronize(c->stream));
            const bool over = count > cap;
            if (sharded) {
                // exchange 2: the tie totals of the open nodes, then the tie list with global columns
                const uint64_t n_local = over ? 0 : count;
                block.assign(1 + n_open + n_local, 0);
                CU_TRY(c, cudaMemcpyAsync(block.data() + 1, d_total, (size_t)n_open * 8, cudaMemcpyDeviceToHost, c->stream));
                CU_TRY(c, cudaMemcpyAsync(block.data() + 1 + n_open, c->cart_list.p, n_local * 8, cudaMemcpyDeviceToHost, c->stream));
                CU_TRY(c, cudaStreamSynchronize(c->stream));
                for (uint64_t i = 0; i < n_local; ++i) block[1 + n_open + i] += sh.off;
                bool any_over = false;
                if (int r = shard_ties(c, sh, count, over, block, (uint64_t)n_open * 8, 8, lists, any_over)) return r;
                if (over) cap = count + count / 4;
                if (any_over) continue;
                h_total.assign(n_open, 0);
                h_list.clear();
                for (const TieList& l : lists) {
                    for (uint32_t i = 0; i < n_open; ++i) {
                        uint64_t x;
                        memcpy(&x, l.p + (size_t)i * 8, 8);
                        h_total[i] += x;
                    }
                    const size_t l0 = h_list.size();
                    h_list.resize(l0 + l.n);
                    memcpy(h_list.data() + l0, l.p + (size_t)n_open * 8, l.n * 8);
                }
                count = h_list.size();
                break;
            }
            if (!over) break;
            cap = count + count / 4;    // the tie list overflowed: grow it and redo the level (nothing was updated)
        }
        if (!sharded) {
            h_best.resize(n_open); h_total.resize(n_open); h_list.resize(count);
            CU_TRY(c, cudaMemcpyAsync(h_best.data(), d_best, (size_t)n_open * 8, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(c, cudaMemcpyAsync(h_total.data(), d_total, (size_t)n_open * 8, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(c, cudaMemcpyAsync(h_list.data(), c->cart_list.p, count * 8, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(c, cudaStreamSynchronize(c->stream));
        }
        // the list comes in the order of the atomics: sorted, each node's entries are its ties in ascending column order
        std::sort(h_list.begin(), h_list.end());
        splits.clear();
        size_t p = 0;
        for (uint32_t i = 0; i < n_open; ++i) {
            size_t e = p;
            while (e < count && (h_list[e] >> 32) == i) ++e;
            if (h_best[i]) {            // else no admissible split: the node stays a leaf
                const grmkm_cart_job& j = jobs[open[i].tree];
                // a pattern matrix's total counts k-mers, its list patterns: the list holds every tie pattern or at
                // least max(1, equiv_cap) of the smallest
                const uint64_t keep = std::min<uint64_t>(c->pat_mult_on ? e - p : h_total[i], j.equiv_cap);
                if (e - p < std::max<uint64_t>(1, keep))
                    return fail(c, GRMKM_E_CUDA, "grmkm_cart_run: the tie list of a node misses members of T");
                std::vector<uint64_t>& eq = c->cart_equiv[open[i].tree];
                grmkm_cart_node& nd = c->cart_nodes[open[i].tree][open[i].node];
                nd.rule = h_list[p] & 0xffffffffULL;
                nd.score = scm_unkey(~h_best[i]);
                nd.equiv_offset = eq.size();
                nd.equiv_count = keep;
                nd.equiv_total = h_total[i];
                for (uint64_t k = 0; k < keep; ++k) eq.push_back(h_list[p + k] & 0xffffffffULL);
                splits.push_back(CartSplit{i, (uint32_t)nd.rule, UINT32_MAX, UINT32_MAX});
            }
            p = e;
        }
        next.clear();
        if (!splits.empty()) {
            const uint32_t n_split = (uint32_t)splits.size();
            // exchange 3 on a slice: the split columns from their owners; gather and split run on their compact matrix
            cols.clear();
            for (const CartSplit& s : splits) cols.push_back(s.j);
            ColumnView v;
            if (int r = column_view(c, sh, cols, v)) return r;
            for (CartSplit& s : splits) s.j = (uint32_t)v.col(s.j);
            CU_TRY(c, cudaMemcpyAsync(d_split, splits.data(), n_split * sizeof(CartSplit), cudaMemcpyHostToDevice, c->stream));
            k_cart_gather<<<(uint32_t)std::min<uint64_t>((n_split + 7) / 8, (uint64_t)c->sm_count * 16), 256, 0, c->stream>>>(
                v.matrix, v.pitch, W, d_masks, d_split, n_split, d_stats);
            CU_TRY(c, cudaGetLastError());
            c->stats.n_launches++;
            h_stats.resize(2 * (size_t)n_split);
            CU_TRY(c, cudaMemcpyAsync(h_stats.data(), d_stats, n_split * 8, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(c, cudaStreamSynchronize(c->stream));
            // children in their parents' order, the present child first: breadth-first numbering
            for (uint32_t k = 0; k < n_split; ++k) {
                const Open o = open[splits[k].src];
                const uint32_t depth = c->cart_nodes[o.tree][o.node].depth + 1;
                const uint32_t a = c->cart_nodes[o.tree][o.node].n_pos, b = c->cart_nodes[o.tree][o.node].n_neg;
                const uint32_t pl = h_stats[2 * k], nl = h_stats[2 * k + 1];
                const uint32_t pc = add_node(o.tree, depth, pl, nl), ac = add_node(o.tree, depth, a - pl, b - nl);
                c->cart_nodes[o.tree][o.node].present_child = pc;
                c->cart_nodes[o.tree][o.node].absent_child = ac;
                if (opens(o.tree, depth, pl, nl)) { splits[k].dst_present = (uint32_t)next.size(); next.push_back({o.tree, pc}); }
                if (opens(o.tree, depth, a - pl, b - nl)) { splits[k].dst_absent = (uint32_t)next.size(); next.push_back({o.tree, ac}); }
            }
            if (!next.empty()) {
                ENSURE(c, c->cart_masks[cur ^ 1], next.size() * 2 * W * 8);
                CU_TRY(c, cudaMemcpyAsync(d_split, splits.data(), n_split * sizeof(CartSplit), cudaMemcpyHostToDevice, c->stream));
                const uint64_t nw = (uint64_t)n_split * W;
                k_cart_split<<<(uint32_t)std::min<uint64_t>((nw + 255) / 256, (uint64_t)c->sm_count * 8), 256, 0, c->stream>>>(
                    v.matrix, v.pitch, W, d_masks, d_split, n_split, (unsigned long long*)c->cart_masks[cur ^ 1].p);
                CU_TRY(c, cudaGetLastError());
                c->stats.n_launches++;
                cur ^= 1;
            }
        }
        open.swap(next);
    }
    CU_TRY(c, cudaStreamSynchronize(c->stream));
    return GRMKM_OK;
}

}  // namespace

extern "C" {

int grmkm_cart_run(grmkm_ctx* c, uint32_t n_trees, const grmkm_cart_job* jobs, const uint64_t* blacklist, uint64_t n_blacklist) {
    return cart_run(c, n_trees, jobs, blacklist, n_blacklist, nullptr,
                    "the result is one owner's slice of a multi-GPU build: its best split is not the answer");
}

int grmkm_cart_run_sharded(grmkm_ctx* c, uint32_t n_trees, const grmkm_cart_job* jobs, const uint64_t* blacklist,
                           uint64_t n_blacklist, const grmkm_shard* shard) {
    return cart_run(c, n_trees, jobs, blacklist, n_blacklist, shard, nullptr);
}

int grmkm_cart_result(grmkm_ctx* c, uint32_t tree, grmkm_cart_node* nodes, uint64_t nodes_cap, uint64_t* n_nodes,
                      uint64_t* equivalent, uint64_t equiv_cap, uint64_t* n_equivalent) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (tree >= c->cart_nodes.size()) return fail(c, GRMKM_E_INVALID, "no such tree in the last grmkm_cart_run");
    return copy_result(c, c->cart_nodes[tree], c->cart_equiv[tree], nodes, nodes_cap, n_nodes, equivalent, equiv_cap,
                       n_equivalent, "cart result buffers too small");
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// grmkm_query: the inputs' genome rows against a set of k-mers, without a build
// ------------------------------------------------------------------------------------------------
namespace {

// device memory of one row range: its presence plane (or counters) and its word rows in the caller's column order.
// Over this, the query runs as consecutive row ranges, each a pass over its own rows' inputs only.
constexpr uint64_t kQueryBudget = 1ULL << 30;

uint64_t canonical_kmer(uint64_t x, uint32_t k) {
    uint64_t rc = 0, f = x;
    for (uint32_t i = 0; i < k; ++i) { rc = (rc << 2) | ((f & 3) ^ 2); f >>= 2; }
    return std::min(x, rc);
}

int query_impl(grmkm_ctx* c, const uint64_t* kmers, uint64_t n, uint64_t* dst, uint32_t G, grmkm_query_stats& qs) {
    CU_TRY(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const uint32_t k = c->cfg.k;
    for (cudaEvent_t& e : c->ev_query) if (!e) CU_TRY(c, cudaEventCreate(&e));
    CU_TRY(c, cudaEventRecord(c->ev_query[0], st));

    // ---- distinct canonical keys in ascending hash order (the build's column order) and the caller's column -> key
    std::vector<std::pair<uint64_t, uint32_t>> hv(n);
    for (uint64_t i = 0; i < n; ++i) hv[i] = {khash(canonical_kmer(kmers[i], k)), (uint32_t)i};
    std::sort(hv.begin(), hv.end());
    std::vector<uint64_t> keys;
    std::vector<uint32_t> col(n);
    for (uint64_t j = 0; j < n; ++j) {
        if (j == 0 || hv[j].first != hv[j - 1].first) keys.push_back(kunhash(hv[j].first));
        col[hv[j].second] = (uint32_t)(keys.size() - 1);
    }
    std::vector<std::pair<uint64_t, uint32_t>>().swap(hv);
    const uint64_t Qd = keys.size();
    qs.n_queries = Qd;
    // ---- open addressing, linear probing, home slot = top bits of fmix64 (grmkm_query.cuh).  kEmptyKey (UINT64_MAX)
    // is never a canonical k-mer: below k = 32 every k-mer is < 2^62, and at k = 32 UINT64_MAX is all-G, whose reverse
    // complement all-C is smaller.
    const uint32_t slot_bits = std::max(1u, ceil_log2(2 * Qd));
    const uint64_t slots = 1ULL << slot_bits;
    std::vector<uint64_t> tk(slots, kEmptyKey);
    std::vector<uint32_t> ti(slots, 0);
    for (uint64_t q = 0; q < Qd; ++q) {
        uint64_t s = fmix64(keys[q]) >> (64 - slot_bits);
        while (tk[s] != kEmptyKey) s = (s + 1) & (slots - 1);
        tk[s] = keys[q]; ti[s] = (uint32_t)q;
    }
    const size_t tab_bytes = slots * 12 + n * 4 + 16;
    ENSURE(c, c->qry, tab_bytes);
    unsigned long long* d_keys = (unsigned long long*)c->qry.p;
    unsigned long long* d_totals = d_keys + slots;
    uint32_t* d_idx = (uint32_t*)(d_totals + 2);
    uint32_t* d_col = d_idx + slots;
    CU_TRY(c, cudaMemcpyAsync(d_keys, tk.data(), slots * 8, cudaMemcpyHostToDevice, st));
    CU_TRY(c, cudaMemsetAsync(d_totals, 0, 16, st));
    CU_TRY(c, cudaMemcpyAsync(d_idx, ti.data(), slots * 4, cudaMemcpyHostToDevice, st));
    CU_TRY(c, cudaMemcpyAsync(d_col, col.data(), n * 4, cudaMemcpyHostToDevice, st));

    QueryJob qj;
    qj.count = c->cfg.min_abundance > 1;
    qj.smem = Qd <= kQuerySmemKeys && !getenv("GRMKM_QUERY_GLOBAL");
    qj.smem_bytes = qj.smem ? slots * 8 : 0;
    {
        void (*kern)(QueryScanParams) = qj.smem ? (qj.count ? k_query_scan<true, true> : k_query_scan<true, false>)
                                                : (qj.count ? k_query_scan<false, true> : k_query_scan<false, false>);
        if (qj.smem) CU_TRY(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qj.smem_bytes));
        int occ = 0;
        CU_TRY(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kQsThreads, qj.smem_bytes));
        qj.ctas_per_sm = (uint32_t)std::max(1, occ);
    }
    qj.sp.k = k; qj.sp.keys = d_keys; qj.sp.idx = d_idx; qj.sp.slot_bits = slot_bits; qj.sp.qd = Qd; qj.sp.totals = d_totals;

    // ---- row ranges: the plane (or counters) and the gathered word rows of one range stay within kQueryBudget
    uint64_t rows_per;
    if (!qj.count) rows_per = 64 * std::max<uint64_t>(1, kQueryBudget / ((Qd + n) * 8));
    else rows_per = kQueryBudget > 2 * n * 8 ? std::max<uint64_t>(1, (kQueryBudget - 2 * n * 8) / (Qd * 4 + n * 8 / 64 + 1)) : 1;
    if (const char* e = getenv("GRMKM_QUERY_ROWS")) {
        const uint64_t v = (uint64_t)std::max(1LL, atoll(e));
        rows_per = qj.count ? v : (v + 63) / 64 * 64;          // presence ranges are whole word rows
    }
    rows_per = std::min<uint64_t>(rows_per, G);
    const uint32_t n_ranges = (uint32_t)((G + rows_per - 1) / rows_per);
    if (n_ranges > 1)
        std::stable_sort(c->inputs.begin(), c->inputs.end(), [](const Input& a, const Input& b) { return a.row < b.row; });
    const InputTable tab = tabulate_inputs(c);
    const uint32_t F = (uint32_t)c->inputs.size();
    Geo geo;
    geo.G = G; geo.W = (G + 63) / 64;

    std::vector<uint64_t> boundary(n);          // a word row shared by two counter ranges: ORed on the host
    uint32_t next_word = 0;                     // word rows of dst below this have been written
    uint64_t sc[S_COUNT];
    for (uint32_t r0 = 0; r0 < G; r0 += (uint32_t)rows_per) {
        const uint32_t nr = (uint32_t)std::min<uint64_t>(rows_per, G - r0);
        const uint32_t w0 = r0 >> 6, w1 = ((r0 + nr - 1) >> 6) + 1, nw = w1 - w0;
        const uint32_t f0 = n_ranges > 1 ? tab.first_file[r0] : 0, f1 = n_ranges > 1 ? tab.first_file[r0 + nr] : F;
        if (f0 == f1) {                         // rows without input
            if (w1 > next_word) { memset(dst + (uint64_t)std::max(w0, next_word) * n, 0, (uint64_t)(w1 - std::max(w0, next_word)) * n * 8); next_word = w1; }
            continue;
        }
        const uint64_t plane_bytes = qj.count ? (uint64_t)nr * Qd * 4 : (uint64_t)nw * Qd * 8;
        ENSURE(c, c->qplane, plane_bytes);
        ENSURE(c, c->qout, (uint64_t)nw * n * 8);
        CU_TRY(c, cudaMemsetAsync(c->qplane.p, 0, plane_bytes, st));
        qj.sp.row0 = r0;
        qj.sp.plane = (unsigned long long*)c->qplane.p; qj.sp.counts = (uint32_t*)c->qplane.p;
        Job job; job.f0 = f0; job.f1 = f1; job.row0 = r0; job.n_rows = nr; job.query = &qj;
        JobOut out;
        int rc = run_job(c, geo, job, out);
        if (rc) return rc;
        QueryGatherParams gp{};
        gp.plane = (const unsigned long long*)c->qplane.p; gp.counts = (const uint32_t*)c->qplane.p; gp.col = d_col;
        gp.qd = Qd; gp.n = n; gp.n_words = nw; gp.row0 = r0; gp.n_rows = nr; gp.min_abundance = c->cfg.min_abundance;
        gp.out = (unsigned long long*)c->qout.p;
        const uint32_t ggrid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(((uint64_t)nw * n + 255) / 256, (uint64_t)c->sm_count * 8));
        if (qj.count) k_query_gather<true><<<ggrid, 256, 0, st>>>(gp);
        else k_query_gather<false><<<ggrid, 256, 0, st>>>(gp);
        CU_TRY(c, cudaGetLastError());
        CU_TRY(c, cudaMemcpyAsync(sc, c->scalars.p, sizeof sc, cudaMemcpyDeviceToHost, st));
        uint32_t wd = w0;
        if (w0 < next_word) {                   // only counter ranges share a word row with the range before
            CU_TRY(c, cudaMemcpyAsync(boundary.data(), c->qout.p, n * 8, cudaMemcpyDeviceToHost, st));
            wd = w0 + 1;
        }
        if (w1 > wd) CU_TRY(c, cudaMemcpyAsync(dst + (uint64_t)wd * n, (const uint64_t*)c->qout.p + (uint64_t)(wd - w0) * n,
                                               (uint64_t)(w1 - wd) * n * 8, cudaMemcpyDeviceToHost, st));
        CU_TRY(c, cudaStreamSynchronize(st));
        if (wd > w0) for (uint64_t i = 0; i < n; ++i) dst[(uint64_t)w0 * n + i] |= boundary[i];
        next_word = w1;
        qs.n_records += sc[S_N_RECORDS];
        qs.n_bases += sc[S_STREAM_TOTAL] - sc[S_N_RECORDS];
    }
    uint64_t tot[2] = {0, 0};
    CU_TRY(c, cudaMemcpyAsync(tot, d_totals, 16, cudaMemcpyDeviceToHost, st));
    CU_TRY(c, cudaEventRecord(c->ev_query[1], st));
    CU_TRY(c, cudaStreamSynchronize(st));
    qs.n_windows = tot[0]; qs.n_hits = tot[1]; qs.n_jobs = n_ranges;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_query[0], c->ev_query[1]) == cudaSuccess) qs.ms = ms; else cudaGetLastError();
    return GRMKM_OK;
}

}  // namespace

extern "C" {

int grmkm_query(grmkm_ctx* c, const uint64_t* kmers, uint64_t n_kmers, uint64_t* dst, uint64_t cap, grmkm_query_stats* stats) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (stats && stats->struct_size != sizeof(grmkm_query_stats))
        return fail(c, GRMKM_E_INVALID, "stats->struct_size must be sizeof(grmkm_query_stats)");
    if (c->cfg.flags & GRMKM_FLAG_COUNTS) return fail(c, GRMKM_E_INVALID, "a pooled count table has no genome rows to query");
    if (n_kmers && !kmers) return fail(c, GRMKM_E_INVALID, "null k-mer list");
    if (n_kmers > 0xFFFFFFFFULL) return fail(c, GRMKM_E_INVALID, "at most 2^32 - 1 k-mers in one query");
    const uint32_t k = c->cfg.k;
    if (k < 32)
        for (uint64_t i = 0; i < n_kmers; ++i)
            if (kmers[i] >> (2 * k))
                return fail(c, GRMKM_E_INVALID, "k-mer " + std::to_string(i) + " is not below 4^k (k = " + std::to_string(k) + ")");
    uint32_t G = c->n_genomes_decl;
    grmkm_query_stats qs{};
    qs.struct_size = sizeof qs;
    for (const Input& in : c->inputs) { G = std::max(G, in.row + 1); qs.n_input_bytes += in.len; }
    const uint64_t need = (uint64_t)((G + 63) / 64) * n_kmers;
    if (cap < need) return fail(c, GRMKM_E_CAPACITY, "dst holds fewer than ceil(G/64) x n_kmers words");
    if (need && !dst) return fail(c, GRMKM_E_INVALID, "null dst");
    if (need) {
        NvtxRange nv("grmkm_query");
        const int r = query_impl(c, kmers, n_kmers, dst, G, qs);
        if (r != GRMKM_OK) {
            // nothing in flight reads the caller's buffers any more, and no side-stream clear is counted on
            const std::string msg = c->err;
            cudaStreamSynchronize(c->stream);
            if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
            if (c->aux_stream) cudaStreamSynchronize(c->aux_stream);
            cudaGetLastError();
            c->pre_pending = false;
            c->err = msg;
            return r;
        }
    }
    if (stats) *stats = qs;
    return GRMKM_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// grmkm_eval_run: fitted models scored on example sets, counts only
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(EvalNode) == sizeof(grmkm_eval_node), "EvalNode mirrors grmkm_eval_node");

namespace {

// The jobs scored on this rank's matrix; sh: the whole matrix (no exchange) or one slice of it.  Sharded, the columns
// of the jobs' rules and split k-mers are exchanged once and every rank scores all jobs on their compact matrix.
int eval_run(grmkm_ctx* c, uint32_t n_jobs, const grmkm_eval_job* jobs, uint32_t* counts, uint64_t cap,
             const grmkm_shard* shard, const char* refusal) {
    Shard sh;
    if (int r = run_shard(c, shard, refusal, sh)) return r;
    const uint64_t UG = sh.total;
    const uint32_t W = c->W;
    uint64_t pairs = 0, n_rules = 0, n_nodes = 0;
    auto validate = [&]() -> int {
        if (int r = check_run(c, sh, nullptr, nullptr, 0)) return r;
        if (n_jobs && !jobs) return fail(c, GRMKM_E_INVALID, "null jobs");
        std::vector<uint8_t> has_parent;
        for (uint32_t i = 0; i < n_jobs; ++i) {
            const grmkm_eval_job& j = jobs[i];
            const std::string at = " (job " + std::to_string(i) + ")";
            if (j.struct_size != sizeof(grmkm_eval_job)) return fail(c, GRMKM_E_INVALID, "job struct_size is not sizeof(grmkm_eval_job)" + at);
            if (j.reserved != 0) return fail(c, GRMKM_E_INVALID, "reserved must be 0" + at);
            if (j.kind > GRMKM_EVAL_CART) return fail(c, GRMKM_E_INVALID, "unknown job kind" + at);
            if (j.n_items >= 0xFFFFFFFFULL) return fail(c, GRMKM_E_INVALID, "at most 2^32 - 2 rules or nodes per job" + at);
            if (j.kind == GRMKM_EVAL_SCM) {
                if (j.model_type > GRMKM_SCM_DISJUNCTION) return fail(c, GRMKM_E_INVALID, "unknown model type" + at);
                if (j.n_items && !j.rules) return fail(c, GRMKM_E_INVALID, "null rules" + at);
                for (uint64_t r = 0; r < j.n_items; ++r)
                    if (j.rules[r] >= 2 * UG) return fail(c, GRMKM_E_INVALID, "rule index >= 2 x n_kmers" + at);
                n_rules += j.n_items;
                pairs += j.n_items + 1;
            } else {
                if (j.model_type != 0) return fail(c, GRMKM_E_INVALID, "model_type of a tree must be 0" + at);
                if (j.n_items == 0) return fail(c, GRMKM_E_INVALID, "a tree has at least its root node" + at);
                if (!j.nodes) return fail(c, GRMKM_E_INVALID, "null nodes" + at);
                const uint64_t n = j.n_items;
                has_parent.assign(n, 0);
                for (uint64_t k = 0; k < n; ++k) {
                    const grmkm_eval_node& e = j.nodes[k];
                    if (e.kmer == UINT64_MAX) continue;
                    const std::string nat = " (job " + std::to_string(i) + ", node " + std::to_string(k) + ")";
                    if (e.kmer >= UG) return fail(c, GRMKM_E_INVALID, "split k-mer >= n_kmers" + nat);
                    for (uint32_t ch : {e.present_child, e.absent_child}) {
                        if (ch <= k || ch >= n) return fail(c, GRMKM_E_INVALID, "a child index must be above its parent's and below n" + nat);
                        if (has_parent[ch]) return fail(c, GRMKM_E_INVALID, "node " + std::to_string(ch) + " has two parents" + at);
                        has_parent[ch] = 1;
                    }
                }
                n_nodes += n;
                pairs += n;
            }
            if (int r = check_examples(c, j.pos, j.neg, at)) return r;
        }
        if (cap < 2 * pairs) return fail(c, GRMKM_E_CAPACITY, "counts holds fewer than 2 x the count pairs of the jobs");
        if (pairs && !counts) return fail(c, GRMKM_E_INVALID, "null counts");
        return GRMKM_OK;
    };
    if (int r = shard_agree(c, sh, validate())) return r;
    if (!pairs) return GRMKM_OK;

    NvtxRange nv("grmkm_eval_run");
    std::vector<EvalJobArg> args(n_jobs);
    std::vector<uint64_t> h_rules, h_masks((size_t)n_jobs * 2 * W);
    std::vector<grmkm_eval_node> h_nodes;
    h_rules.reserve(n_rules);
    h_nodes.reserve(n_nodes);
    uint64_t out = 0;
    for (uint32_t i = 0; i < n_jobs; ++i) {
        const grmkm_eval_job& j = jobs[i];
        const bool scm = j.kind == GRMKM_EVAL_SCM;
        args[i] = EvalJobArg{scm ? EVAL_SCM : EVAL_CART, (uint32_t)(scm && j.model_type == GRMKM_SCM_CONJUNCTION),
                             (uint32_t)j.n_items, 0, scm ? h_rules.size() : h_nodes.size(), out};
        if (scm) h_rules.insert(h_rules.end(), j.rules, j.rules + j.n_items);
        else h_nodes.insert(h_nodes.end(), j.nodes, j.nodes + j.n_items);
        out += scm ? j.n_items + 1 : j.n_items;
        if (W) {
            memcpy(h_masks.data() + (size_t)i * 2 * W, j.pos, (size_t)W * 8);
            memcpy(h_masks.data() + (size_t)i * 2 * W + W, j.neg, (size_t)W * 8);
        }
    }
    CU_TRY(c, cudaSetDevice(c->device));
    // on a slice, the columns of every rule and split k-mer from their owners; the jobs name them by their compact index
    std::vector<uint64_t> cols;
    for (uint64_t r : h_rules) cols.push_back(r % UG);
    for (const grmkm_eval_node& e : h_nodes) if (e.kmer != UINT64_MAX) cols.push_back(e.kmer);
    ColumnView v;
    if (int r = column_view(c, sh, std::move(cols), v)) return r;
    for (uint64_t& r : h_rules) r = v.rule(r, UG);
    for (grmkm_eval_node& e : h_nodes) if (e.kmer != UINT64_MAX) e.kmer = v.col(e.kmer);
    auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t o_args = 0, o_rules = al((size_t)n_jobs * sizeof(EvalJobArg)), o_nodes = o_rules + al(n_rules * 8),
                 o_masks = o_nodes + al(n_nodes * sizeof(EvalNode)), o_cnt = o_masks + al(h_masks.size() * 8),
                 total = o_cnt + pairs * 8;
    ENSURE(c, c->eval, total);
    uint8_t* base = (uint8_t*)c->eval.p;
    cudaStream_t st = c->stream;
    CU_TRY(c, cudaMemcpyAsync(base + o_args, args.data(), (size_t)n_jobs * sizeof(EvalJobArg), cudaMemcpyHostToDevice, st));
    if (n_rules) CU_TRY(c, cudaMemcpyAsync(base + o_rules, h_rules.data(), n_rules * 8, cudaMemcpyHostToDevice, st));
    if (n_nodes) CU_TRY(c, cudaMemcpyAsync(base + o_nodes, h_nodes.data(), n_nodes * sizeof(EvalNode), cudaMemcpyHostToDevice, st));
    if (!h_masks.empty()) CU_TRY(c, cudaMemcpyAsync(base + o_masks, h_masks.data(), h_masks.size() * 8, cudaMemcpyHostToDevice, st));
    CU_TRY(c, cudaMemsetAsync(base + o_cnt, 0, pairs * 8, st));
    const uint32_t warps_per_cta = kEvalThreads / 32;
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((n_jobs + warps_per_cta - 1) / warps_per_cta,
                                                                              (uint64_t)c->sm_count * 8));
    k_eval<<<grid, kEvalThreads, 0, st>>>(v.matrix, v.U, v.pitch, W, (const EvalJobArg*)(base + o_args),
                                          n_jobs, (const unsigned long long*)(base + o_rules), (const EvalNode*)(base + o_nodes),
                                          (const unsigned long long*)(base + o_masks), (uint32_t*)(base + o_cnt));
    CU_TRY(c, cudaGetLastError());
    c->stats.n_launches++;
    CU_TRY(c, cudaMemcpyAsync(counts, base + o_cnt, pairs * 8, cudaMemcpyDeviceToHost, st));
    CU_TRY(c, cudaStreamSynchronize(st));
    return GRMKM_OK;
}

}  // namespace

extern "C" {

int grmkm_eval_run(grmkm_ctx* c, uint32_t n_jobs, const grmkm_eval_job* jobs, uint32_t* counts, uint64_t cap) {
    return eval_run(c, n_jobs, jobs, counts, cap, nullptr,
                    "the result is one owner's slice of a multi-GPU build: it holds some k-mers only");
}

int grmkm_eval_run_sharded(grmkm_ctx* c, uint32_t n_jobs, const grmkm_eval_job* jobs, uint32_t* counts, uint64_t cap,
                           const grmkm_shard* shard) {
    return eval_run(c, n_jobs, jobs, counts, cap, shard, nullptr);
}

int grmkm_copy_columns(grmkm_ctx* c, const uint64_t* idx, uint64_t n, uint64_t* dst, uint64_t cap) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build or grmkm_load_result first");
    if (n && !idx) return fail(c, GRMKM_E_INVALID, "null column indices");
    if (n > 0xFFFFFFFFULL) return fail(c, GRMKM_E_INVALID, "at most 2^32 - 1 columns in one call");
    for (uint64_t i = 0; i < n; ++i)
        if (idx[i] >= c->U) return fail(c, GRMKM_E_INVALID, "column index >= n_kmers");
    if (cap < n * c->W) return fail(c, GRMKM_E_CAPACITY, "dst holds fewer than n_words x n words");
    if (n && c->W && !dst) return fail(c, GRMKM_E_INVALID, "null dst");
    CU_TRY(c, cudaSetDevice(c->device));
    return pack_columns(c, idx, n, dst);
}

// ------------------------------------------------------------------------------------------------
// grmkm_patterns: the distinct presence patterns of the result (grmkm_patterns.cuh)
// ------------------------------------------------------------------------------------------------
int grmkm_patterns(grmkm_ctx* c, const uint8_t* column_class, grmkm_ctx* d, uint32_t* pattern_of_column, uint64_t pattern_cap,
                   uint32_t* members, uint64_t members_cap, uint64_t* member_offsets, uint64_t offsets_cap,
                   grmkm_pattern_stats* stats) {
    if (check_ctx(c)) return GRMKM_E_INVALID;
    if (!d || d == c) return fail(c, GRMKM_E_INVALID, "dst must be a second context, not src");
    if (stats && stats->struct_size != sizeof(grmkm_pattern_stats))
        return fail(c, GRMKM_E_INVALID, "stats struct_size is not sizeof(grmkm_pattern_stats)");
    if (!c->built) return fail(c, GRMKM_E_INVALID, "no result: call grmkm_build or grmkm_load_result first");
    if (c->slice)
        return fail(c, GRMKM_E_UNSUPPORTED, "the result is one owner's slice of a multi-GPU build: patterns across slices are not grouped");
    if (d->device != c->device) return fail(c, GRMKM_E_INVALID, "dst is a context of another device");
    const uint64_t U = c->U;
    const uint32_t W = c->W;
    if (U >= 0xFFFFFFFFULL) return fail(c, GRMKM_E_UNSUPPORTED, "patterns index columns with 32 bits: at most 2^32 - 2 columns");
    if (column_class)
        for (uint64_t j = 0; j < U; ++j)
            if (column_class[j] > 3) return fail(c, GRMKM_E_INVALID, "column class " + std::to_string(column_class[j]) + " > 3");
    uint32_t bits = 64;
    if (const char* e = getenv("GRMKM_PATTERN_HASH_BITS")) bits = (uint32_t)std::min(64, std::max(1, atoi(e)));   // tests: collisions
    CU_TRY(c, cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    NvtxRange nv("grmkm_patterns");

    // scratch, all of it before any launch: U' = max(U, 1) columns, T = the least power of two >= 2 U' table slots
    // (< 4 U'); per column fp 8, slot / flag 4, two active lists 8, head 4, pid 4, pattern 4, member 4, head column 8,
    // multiplicity 4, offset 4, class 1, plus the table's 12 per slot and CUB's scan and sort scratch
    const uint64_t Uc = std::max<uint64_t>(U, 1), U1 = Uc + 1;
    const uint64_t tcap = 1ULL << ceil_log2(2 * Uc);
    size_t scan_tmp = 0, sort_tmp = 0;
    CU_TRY(c, cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (const uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t)U1, st));
    CU_TRY(c, cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                              (const uint32_t*)nullptr, (uint32_t*)nullptr, (uint32_t)Uc, 0, 32, st));
    auto al = [](size_t b) { return (b + 255) & ~size_t(255); };
    const size_t o_fp = 0, o_tkey = o_fp + al(Uc * 8), o_thead = o_tkey + al(tcap * 8), o_slot = o_thead + al(tcap * 4),
                 o_act0 = o_slot + al(U1 * 4), o_act1 = o_act0 + al(Uc * 4), o_head = o_act1 + al(Uc * 4),
                 o_pid = o_head + al(Uc * 4), o_pat = o_pid + al(U1 * 4), o_mem = o_pat + al(Uc * 4),
                 o_heads = o_mem + al(Uc * 4), o_mult = o_heads + al(Uc * 8), o_offs = o_mult + al(U1 * 4),
                 o_cls = o_offs + al(U1 * 4), o_next = o_cls + al(Uc), o_tmp = o_next + 256,
                 total = o_tmp + al(std::max(scan_tmp, sort_tmp));
    ENSURE(c, c->pat, total);
    uint8_t* base = (uint8_t*)c->pat.p;
    unsigned long long* fp = (unsigned long long*)(base + o_fp);
    unsigned long long* tkey = (unsigned long long*)(base + o_tkey);
    uint32_t* thead = (uint32_t*)(base + o_thead);
    uint32_t* slot_of = (uint32_t*)(base + o_slot);     // the rounds: slot of each active column; then the head flags
    uint32_t* act[2] = {(uint32_t*)(base + o_act0), (uint32_t*)(base + o_act1)};   // then the sort's values in / keys out
    uint32_t* head_of = (uint32_t*)(base + o_head);
    uint32_t* pid = (uint32_t*)(base + o_pid);
    uint32_t* pat_of = (uint32_t*)(base + o_pat);
    uint32_t* mem = (uint32_t*)(base + o_mem);
    unsigned long long* heads = (unsigned long long*)(base + o_heads);
    uint32_t* mult = (uint32_t*)(base + o_mult);
    uint32_t* offs = (uint32_t*)(base + o_offs);
    uint8_t* cls = column_class ? base + o_cls : nullptr;
    unsigned int* n_next = (unsigned int*)(base + o_next);
    void* tmp = base + o_tmp;

    cudaEvent_t ev[2] = {nullptr, nullptr};
    CU_TRY(c, cudaEventCreate(&ev[0]));
    CU_TRY(c, cudaEventCreate(&ev[1]));
    struct EvGuard { cudaEvent_t* e; ~EvGuard() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } ev_guard{ev};
    CU_TRY(c, cudaEventRecord(ev[0], st));
    const unsigned long long* m = (const unsigned long long*)c->matrix.p;
    auto grid_of = [&](uint64_t n) { return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>((n + 255) / 256, (uint64_t)c->sm_count * 16)); };
    uint32_t rounds = 0;
    uint32_t P = 0;
    if (U) {
        if (cls) CU_TRY(c, cudaMemcpyAsync(cls, column_class, U, cudaMemcpyHostToDevice, st));
        k_pat_hash<<<grid_of(U), 256, 0, st>>>(m, c->pitch, W, (uint32_t)U, cls, bits, fp);
        CU_TRY(c, cudaGetLastError());
        c->stats.n_launches++;
        // rounds: every column of the round settles or moves to the next one, whose table has no settled head
        uint32_t n = (uint32_t)U;
        const uint32_t* cur = nullptr;          // round 1: all columns
        for (int nxt = 0; n; ++rounds) {
            const uint64_t T = 1ULL << ceil_log2(2 * (uint64_t)n);
            CU_TRY(c, cudaMemsetAsync(tkey, 0xff, T * 8, st));
            CU_TRY(c, cudaMemsetAsync(thead, 0xff, T * 4, st));
            CU_TRY(c, cudaMemsetAsync(n_next, 0, 4, st));
            k_pat_insert<<<grid_of(n), 256, 0, st>>>(cur, n, fp, tkey, thead, T - 1, slot_of);
            k_pat_verify<<<grid_of(n), 256, 0, st>>>(m, c->pitch, W, cls, cur, n, slot_of, thead, head_of, act[nxt], n_next);
            CU_TRY(c, cudaGetLastError());
            c->stats.n_launches += 2;
            unsigned int h_next = 0;
            CU_TRY(c, cudaMemcpyAsync(&h_next, n_next, 4, cudaMemcpyDeviceToHost, st));
            CU_TRY(c, cudaStreamSynchronize(st));
            if (h_next >= n) return fail(c, GRMKM_E_CUDA, "grmkm_patterns: a grouping round settled no column");
            n = h_next;
            cur = act[nxt];
            nxt ^= 1;
        }
        // numbering: pid = exclusive scan of the head flags (pid[U] = P)
        k_pat_flags<<<grid_of(U + 1), 256, 0, st>>>(head_of, (uint32_t)U, slot_of);
        CU_TRY(c, cudaGetLastError());
        CU_TRY(c, cub::DeviceScan::ExclusiveSum(tmp, scan_tmp, (const uint32_t*)slot_of, pid, (uint32_t)(U + 1), st));
        CU_TRY(c, cudaMemcpyAsync(&P, pid + U, 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(c, cudaMemsetAsync(mult, 0, (U + 1) * 4, st));
        k_pat_assign<<<grid_of(U), 256, 0, st>>>(head_of, pid, (uint32_t)U, pat_of, act[0], heads, mult);
        CU_TRY(c, cudaGetLastError());
        CU_TRY(c, cudaStreamSynchronize(st));
        // member offsets = exclusive scan of the multiplicities (mult[P] = 0); members = the columns stably sorted by
        // pattern (radix sort over the bits of P - 1: the columns come in ascending order, and stay so in each pattern)
        CU_TRY(c, cub::DeviceScan::ExclusiveSum(tmp, scan_tmp, (const uint32_t*)mult, offs, P + 1, st));
        const int end_bit = (int)std::max<uint32_t>(1, ceil_log2(P));
        size_t need = 0;
        CU_TRY(c, cub::DeviceRadixSort::SortPairs(nullptr, need, (const uint32_t*)pat_of, act[1], (const uint32_t*)act[0], mem,
                                                  (uint32_t)U, 0, end_bit, st));
        if (need > sort_tmp) return fail(c, GRMKM_E_CUDA, "grmkm_patterns: the sort asks for more scratch than was reserved");
        CU_TRY(c, cub::DeviceRadixSort::SortPairs(tmp, sort_tmp, (const uint32_t*)pat_of, act[1], (const uint32_t*)act[0], mem,
                                                  (uint32_t)U, 0, end_bit, st));
        c->stats.n_launches += 3;
    }

    // dst: the P x W matrix of the heads, their k-mers and multiplicities, copied on the device
    if (d->aux_stream) CU_TRY(d, cudaStreamSynchronize(d->aux_stream));
    d->built = false;
    auto dst_ensure = [&](DevBuf& b, size_t bytes) {
        const int r = ensure(d, b, bytes);
        if (r) c->err = d->err;
        return r;
    };
    if (int r = dst_ensure(d->kmers, (size_t)P * 8)) return r;
    if (int r = dst_ensure(d->matrix, (size_t)P * W * 8)) return r;
    if (int r = dst_ensure(d->pat_mult, (size_t)P * 4)) return r;
    if (P) {
        k_gather_columns<<<grid_of((uint64_t)P * 32), 256, 0, st>>>((const unsigned long long*)c->kmers.p, 0, 1, heads, P,
                                                                    (unsigned long long*)d->kmers.p);
        if (W)
            k_gather_columns<<<grid_of((uint64_t)P * 32), 256, 0, st>>>(m, c->pitch, W, heads, P, (unsigned long long*)d->matrix.p);
        CU_TRY(c, cudaGetLastError());
        c->stats.n_launches += W ? 2 : 1;
        CU_TRY(c, cudaMemcpyAsync(d->pat_mult.p, mult, (size_t)P * 4, cudaMemcpyDeviceToDevice, st));
    }
    CU_TRY(c, cudaEventRecord(ev[1], st));
    CU_TRY(c, cudaStreamSynchronize(st));
    float ms = 0.f;
    CU_TRY(c, cudaEventElapsedTime(&ms, ev[0], ev[1]));
    d->U = P; d->W = W; d->G = c->G; d->pitch = P;
    set_result(d, true, true);
    if (stats) { stats->n_rounds = rounds; stats->n_patterns = P; stats->ms = ms; }

    // the mapping to the host: what fits, or GRMKM_E_CAPACITY (dst's result stands either way)
    const bool fits = (pattern_of_column || !U) && pattern_cap >= U && (members || !U) && members_cap >= U &&
                      member_offsets && offsets_cap >= (uint64_t)P + 1;
    if (U && pattern_of_column && pattern_cap >= U)
        CU_TRY(c, cudaMemcpyAsync(pattern_of_column, pat_of, U * 4, cudaMemcpyDeviceToHost, st));
    if (U && members && members_cap >= U) CU_TRY(c, cudaMemcpyAsync(members, mem, U * 4, cudaMemcpyDeviceToHost, st));
    std::vector<uint32_t> h_offs(U ? (size_t)P + 1 : 0);
    if (U && member_offsets && offsets_cap >= (uint64_t)P + 1)
        CU_TRY(c, cudaMemcpyAsync(h_offs.data(), offs, ((size_t)P + 1) * 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(c, cudaStreamSynchronize(st));
    if (member_offsets && offsets_cap >= (uint64_t)P + 1) {
        for (uint32_t p = 0; p < P && U; ++p) member_offsets[p] = h_offs[p];
        member_offsets[P] = U;
    }
    if (!fits) return fail(c, GRMKM_E_CAPACITY, "pattern_of_column / members need U entries, member_offsets P + 1 (P = dst's n_kmers)");
    return GRMKM_OK;
}

}  // extern "C"
