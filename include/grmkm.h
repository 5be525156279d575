/*
 * grmkm.h -- C ABI of libgrmkm.so: the B200-native k-mer matrix builder that
 * replaces the native half of GRM's "genomes -> genome x k-mer matrix" path.
 *
 * The reference has no in-process FFI for this path: it reaches the native
 * code through argv of child processes (SURVEY.md section 8b).  Each entry point
 * below names the reference interface it stands in for; paths are under
 * /root/reference.
 *
 *   multidsk  argv   bin/kover/core/kover/dataset/tools/kmer_count.py:28-37, 44-53
 *   dsk2kover argv   bin/kover/core/kover/dataset/tools/kmer_pack.py:28-36
 *   Ray       argv   src/app.py:1310 + survey.conf grammar src/app.py:3820-3833
 *   dsk       argv   src/app.py:1371-1372
 *
 * Conventions: extern "C", plain pointers and sizes, no exceptions cross the
 * boundary.  Every call returns GRMKM_OK (0) or a negative GRMKM_E_* code; the
 * message is available from grmkm_last_error().  The caller allocates every
 * output buffer and passes its capacity.  A context owns all device memory and
 * is single-owner (not thread safe); several contexts may coexist.  There is
 * NO CPU fallback: without a CUDA device grmkm_create fails with
 * GRMKM_E_NO_DEVICE.
 */
#ifndef GRMKM_H
#define GRMKM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRMKM_ABI_VERSION 15

enum {
    GRMKM_OK = 0,
    GRMKM_E_INVALID = -1,       /* bad argument / bad state                          */
    GRMKM_E_UNSUPPORTED_K = -2, /* k outside 1..32 (reference allows <=128, kover:114) */
    GRMKM_E_NOMEM = -3,         /* host or device allocation failed                  */
    GRMKM_E_CUDA = -4,          /* CUDA runtime error (message has the detail)       */
    GRMKM_E_IO = -5,            /* file could not be read / inflated                 */
    GRMKM_E_CAPACITY = -6,      /* caller buffer too small                           */
    GRMKM_E_NO_DEVICE = -7,     /* no usable CUDA device: there is no CPU fallback   */
    GRMKM_E_UNSUPPORTED = -8    /* e.g. more than 32768 genomes in one context       */
};

enum { GRMKM_FASTA = 0, GRMKM_FASTQ = 1 };

/* cfg.flags */
#define GRMKM_FLAG_COUNTS 32u /* pooled count table (bin/dsk/dsk -file <list> -kmer-size k, src/app.py:1371-1372): every input is
                                 pooled on ONE row, the result has one column per canonical k-mer whose abundance over all inputs
                                 is >= min_abundance, and matrix row 0 holds that abundance (a count, not presence bits) */

typedef struct grmkm_ctx grmkm_ctx;

/*
 * Parameters = the knobs the reference forwards to the native tools:
 *   k               -kmer-size / -kmer-length / "-k"      (kmer_count.py:31, kmer_pack.py:32, app.py:3821)
 *   min_abundance   -abundance-min  (contigs: 1, kmer_count.py:32; reads: user value, :48)
 *   keep_singletons -filter nothing|singleton  (kover:144-147 -> kmer_pack.py:31); Ray mode: 1
 *   input_kind      contigs (.fna, FASTA) or reads (.fastq, FASTQ)  (create.py:278, 399-402)
 */
typedef struct grmkm_config {
    uint32_t struct_size;     /* = sizeof(grmkm_config), for forward compatibility */
    uint32_t k;               /* 1..32 */
    uint32_t min_abundance;   /* >= 1 */
    uint32_t keep_singletons; /* 0: drop k-mers present in exactly one genome */
    uint32_t input_kind;      /* default kind for grmkm_add_genome_* */
    int32_t device;           /* CUDA ordinal; -1 = current device */
    uint32_t bucket_bits;     /* 0 = auto; log2 of the number of hash buckets */
    uint32_t flags;
    void* stream;             /* cudaStream_t to run on; NULL = context-owned stream */
} grmkm_config;

typedef struct grmkm_stats {
    uint64_t n_bases;       /* nucleotide characters in sequence lines             */
    uint64_t n_windows;     /* valid k-mer windows (= records partitioned)         */
    uint64_t n_input_bytes; /* bytes of FASTA/FASTQ text                           */
    uint64_t n_records;     /* FASTA/FASTQ records                                 */
    uint64_t n_kmers;       /* U: columns kept                                     */
    uint64_t n_distinct;    /* distinct canonical k-mers before the singleton filter */
    uint32_t n_words;       /* ceil(G/64)                                          */
    uint32_t n_genomes;     /* G                                                   */
    uint32_t n_buckets;     /* hash buckets used                                   */
    uint32_t n_launches;    /* kernels launched by the last build                  */
    uint64_t h2d_bytes;     /* host->device bytes moved by the last build          */
    uint64_t device_bytes;  /* device memory held by the context                   */
    uint64_t n_splits;      /* bucket sub-range splits (table overflows handled)   */
    uint64_t n_region_overflows; /* builds redone with exact offsets (a bucket region was too small) */
    uint64_t n_units;        /* super-k-mer units scattered                                */
    uint64_t n_unit_entries; /* distinct (unit, 64-genome block) entries after the dedupe  */
    uint64_t n_wide;         /* [hash, presence word] records the distinct units expand to */
    uint32_t n_unit_buckets; /* content-hash buckets of the unit scatter                   */
    uint32_t n_rounds;       /* abundance builds (min_abundance > 1): rounds of genome rows  */
    uint64_t n_solid_records; /* abundance builds: solid (k-mer, round) presence records     */
} grmkm_stats;

/* per-stage device time of the last build, milliseconds (CUDA events on the build stream) */
typedef struct grmkm_times {
    float h2d, parse, pack, count, scatter, abundance, aggregate, sort, total;
    float bounds, dedupe, expand; /* unit path: run boundaries, per-bucket dedupe, expansion to k-mer records */
} grmkm_times;

int grmkm_abi_version(void);
int grmkm_device_count(void);

int grmkm_create(const grmkm_config* cfg, grmkm_ctx** out);
void grmkm_destroy(grmkm_ctx* ctx);
/* ctx may be NULL: message of the last failed grmkm_create on this thread */
const char* grmkm_last_error(const grmkm_ctx* ctx);

/* Forget the inputs (and result) of the previous build; device buffers are kept for reuse. */
int grmkm_reset(grmkm_ctx* ctx);

/*
 * One line of multidsk's "-file" list (create.py:361-362, 482-489): the file(s)
 * of genome `genome_row` (row order = order of genome_identifiers, create.py:334-347).
 * All inputs of one row are pooled.  *_bytes: host memory, borrowed until the
 * build returns.  *_device: device memory on cfg.device, borrowed likewise.
 * *_files: read (and gunzip'ed when the name ends in .gz) by the library.
 */
int grmkm_add_genome_bytes(grmkm_ctx* ctx, uint32_t genome_row, const uint8_t* data, uint64_t n);
int grmkm_add_genome_device(grmkm_ctx* ctx, uint32_t genome_row, const void* dev_data, uint64_t n);
int grmkm_add_genome_files(grmkm_ctx* ctx, uint32_t genome_row, const char* const* paths, int n_paths);
/* The whole "-file" list in one call (the n lines of create.py:361-362 at once): input i belongs to row rows[i],
 * is lens[i] bytes at data[i]; on_device = 0 host memory (as *_bytes), 1 device memory (as *_device). */
int grmkm_add_genomes(grmkm_ctx* ctx, uint32_t n, const uint32_t* rows, const void* const* data, const uint64_t* lens,
                      int on_device);
/* Declare rows without input (trailing empty genomes still get a matrix row). */
int grmkm_set_genome_count(grmkm_ctx* ctx, uint32_t n_genomes);

/*
 * multidsk + dsk2kover in one call: count canonical k-mers per genome, apply
 * min_abundance per genome, merge across genomes, apply the singleton filter,
 * pack 64 genomes per word (bit 63-(g%64) of word g/64, utils.py:144-154).
 * The result stays device-resident until the next reset/build/destroy.
 * min_abundance > 1 (kmer_count.py:48): the genomes are counted a few rows at a time (per-genome abundance
 * counters in the shared-memory tables), the solid presence of every round is kept, and one presence merge
 * over all rounds follows.  GRMKM_FLAG_COUNTS: see the flag.
 */
int grmkm_build(grmkm_ctx* ctx);

int grmkm_dims(const grmkm_ctx* ctx, uint64_t* n_kmers, uint32_t* n_words, uint32_t* n_genomes);
int grmkm_get_stats(const grmkm_ctx* ctx, grmkm_stats* out);
int grmkm_stage_times(const grmkm_ctx* ctx, grmkm_times* out);

/* canonical k-mers as integers (A0 C1 T2 G3, first base most significant); cap in elements.
 * Column order: ascending grmkm_hash64(k-mer) = k-mer * 0x9E3779B97F4A7C15 mod 2^64 (the order the hash
 * partitions come out in, identical for any GPU count; the reference's own column order is the unspecified
 * partition order of DSK, SURVEY.md 8a-8). */
int grmkm_copy_kmers_packed(grmkm_ctx* ctx, uint64_t* dst, uint64_t cap);
/* kmer_sequences: U x k bytes, upper-case, no terminator (create.py:216-220, ds.py:84); cap in bytes */
int grmkm_copy_kmer_strings(grmkm_ctx* ctx, char* dst, uint64_t cap);
/* kmer_matrix: row-major n_words x U (create.py:224-230); cap in elements */
int grmkm_copy_matrix(grmkm_ctx* ctx, uint64_t* dst, uint64_t cap);
/*
 * Ray Surveyor KmerMatrix.tsv (consumer grammar create.py:121-137,241-264):
 * "kmers\t<name_1>...\n" then fixed-width rows "<kmer>\t<0|1>...\n".
 * dst may be NULL to query the size (returned in *written with GRMKM_E_CAPACITY).
 */
int grmkm_format_tsv(grmkm_ctx* ctx, const char* const* names, char* dst, uint64_t cap, uint64_t* written);

/*
 * The result in page-locked host memory owned by the context: one device->host copy at PCIe speed (a copy
 * into pageable caller memory runs 10x slower).  kmers[U], matrix[n_words][U] row-major; the pointers stay
 * valid until the next build / reset / destroy of this context.
 */
int grmkm_host_result(grmkm_ctx* ctx, const uint64_t** kmers, const uint64_t** matrix);

/*
 * Kernels over the finished, device-resident result.
 *
 * grmkm_result_checksum: order-independent 128-bit digest of the columns (k-mer + its words); the digests of the
 *   ranks' slices of a multi-GPU build add up (mod 2^64 per lane) to the digest of the one-GPU matrix.
 * grmkm_sum_rows: KmerRuleClassifications.sum_rows (bin/kover/core/kover/learning/common/rules.py:201-267 with
 *   popcount.pyx:76-95): dst[j] = sum over word rows w of popcount(matrix[w][j] & row_mask[w]); row_mask has
 *   n_words words, example (genome row) g at bit 63-(g%64) of word g/64 (build_row_mask, rules.py:209-222).
 * grmkm_gram: G x G matrix of shared columns, dst[a*G+b] = #columns present in genomes a and b (the similarity
 *   matrix Ray Surveyor prints beside the k-mer matrix, src/app.py:1310).
 */
int grmkm_result_checksum(grmkm_ctx* ctx, uint64_t out[2]);
int grmkm_sum_rows(grmkm_ctx* ctx, const uint64_t* row_mask, uint32_t n_mask_words, uint32_t* dst, uint64_t cap);
int grmkm_gram(grmkm_ctx* ctx, uint64_t* dst, uint64_t cap);

/*
 * from_tsv's bit packer on the GPU (dataset/create.py:241-271 with utils.py:133-156): body = n_rows fixed-width
 * rows "<k-mer>\t<c_0>\t<c_1>...\n" of a Ray Surveyor KmerMatrix.tsv (host memory, row_width = k + 2 x
 * n_tsv_cols + 1); matrix row g takes TSV column sel[g]; dst = row-major ceil(n_genomes/64) x n_rows words
 * (host memory).  A cell other than '0' / '1' fails with GRMKM_E_INVALID (create.py:121-137: binary matrix).
 * Needs no build; any context of the device will do.
 */
int grmkm_tsv_pack(grmkm_ctx* ctx, const uint8_t* body, uint64_t n_rows, uint32_t row_width, uint32_t k,
                   uint32_t n_tsv_cols, uint32_t n_genomes, const uint32_t* sel, uint64_t* dst, uint64_t cap);

/* Device pointers of the result for callers that stay on the GPU: kmers[U] and the matrix, whose word row w starts at
 * d_matrix + w * pitch_words (pitch_words >= U: the columns are written at their final place while their number is
 * still unknown, so the rows are spaced by the build's capacity; the host copies above deliver rows U words apart). */
int grmkm_device_result(const grmkm_ctx* ctx, const uint64_t** d_kmers, const uint64_t** d_matrix, uint64_t* pitch_words);

/*
 * Bench/test utility: materialise the synthetic FASTA of BASELINE.md section 4 /
 * SURVEY.md section 8d on the device.  layout = host table produced by
 * genomic-resistance-mapping-grm-_b200/synth.py (see grmkm_synth_genome there).
 */
int grmkm_synth_fasta_device(grmkm_ctx* ctx, const void* layout, uint64_t layout_bytes, void* dev_dst,
                             uint64_t dst_bytes);

/*
 * Multi-GPU (one context per process/GPU, SURVEY.md section 8e).  The exchange is either fused into the export
 * (grmkm_export_partials_peers: NVLink stores into the owners' receive buffers) or done by the host layer with
 * an all-to-all over NCCL on the buffer grmkm_export_partials fills.
 *
 * grmkm_build_partial: local stages only.  Produces partial columns
 * (hashed k-mer, n_local_words words) grouped by owner rank = hash range,
 * owner r holding buckets [r*B/P, (r+1)*B/P).  counts[P] receives the number of
 * partial columns per owner.  Export copies them, owner-major, as
 * u64 records of (1 + n_local_words) words into caller device memory.
 *
 * grmkm_merge_partials: owner side.  parts = device buffer with the received
 * partial columns of all P sources back to back (source-major), src_counts[P]
 * their lengths, src_words[P] the words per source; source s contributes matrix
 * word rows [word_offset_s, word_offset_s + src_words[s]).  Applies the
 * singleton filter on the full popcount and leaves this owner's slice of the
 * result in the context (dims/copy_* as after grmkm_build).
 */
int grmkm_build_partial(grmkm_ctx* ctx, uint32_t n_ranks, uint64_t* counts);
/* All ranks must partition the hash space identically: read this rank's automatic choice for
 * the inputs added so far, agree on the maximum over ranks, set it before grmkm_build_partial (which refuses
 * n_ranks > 1 without it) and keep it set for grmkm_merge_partials: the owners' hash ranges are cut on that grid. */
int grmkm_plan_bucket_bits(grmkm_ctx* ctx, uint32_t* bits);
int grmkm_set_bucket_bits(grmkm_ctx* ctx, uint32_t bits);
int grmkm_export_partials(grmkm_ctx* ctx, void* dev_dst, uint64_t dst_bytes);
/* The export fused with the all-to-all: owner d's slice of the partial columns is stored straight into rank d's
 * receive buffer (peer_dst[d], peer-accessible device memory, e.g. torch symmetric memory) at word offset
 * peer_word_off[d] -- over NVLink, no send buffer and no NCCL send/recv (Ray's message routing, src/app.py:1310).
 * Asynchronous on the context's stream; the ranks synchronise (barrier) before anybody merges. */
int grmkm_export_partials_peers(grmkm_ctx* ctx, uint32_t n_ranks, void* const* peer_dst, const uint64_t* peer_word_off);
/* This context's rank among the exporters (default: its device index).  Only staggers the order in which the export walks
 * the owners -- rank r starts with owner r + 1 -- so that the P exporters store into P different receivers at any moment
 * (the hash-routed message rounds of `mpiexec -n 4 Ray`, src/app.py:1310); the result does not depend on it. */
int grmkm_set_exchange_rank(grmkm_ctx* ctx, uint32_t rank);
int grmkm_merge_partials(grmkm_ctx* ctx, const void* dev_parts, uint32_t n_ranks, uint32_t rank,
                         const uint64_t* src_counts, const uint32_t* src_words, uint32_t total_genomes);

/*
 * An existing matrix as the context's result (a .kover file's kmer_matrix and its k-mers): kmers[n_kmers] packed as
 * grmkm_copy_kmers_packed returns them, matrix row-major ceil(n_genomes / 64) x n_kmers (host memory).  Every result-side
 * call then works on it as on a build.  Set bits at rows >= n_genomes: GRMKM_E_INVALID; n_genomes > 32768:
 * GRMKM_E_UNSUPPORTED.
 */
int grmkm_load_result(grmkm_ctx* ctx, const uint64_t* kmers, const uint64_t* matrix, uint64_t n_kmers, uint32_t n_genomes);

/*
 * Set Covering Machine (kover learning/learners/scm.py) on the resident matrix, many fits at once.  Rule r < U is
 * "k-mer r present", rule U + r its absence twin.  Per fit (disjunction: P0 and N0 swapped first), P = P0, N = N0;
 * while |N| > 0 and fewer than max_rules rules: over the rules not blacklisted, e = #P examples the rule outputs 0 on,
 * c = #N examples it outputs 0 on, u = (double)c - p * (double)e (product rounded, then difference); u* = max u;
 * T = {u == u*, c > 0 or e > 0} (empty: stop); tiebreak: keep the T members of least risk (#P0 outputs 0 + #N0
 * outputs 1); the rule is min T; P and N keep the examples it outputs 1 on.  Every greedy step of all fits is one
 * pass over the matrix on the device; only the steps and the sets T cross PCIe.
 */
enum { GRMKM_SCM_CONJUNCTION = 0, GRMKM_SCM_DISJUNCTION = 1 };

typedef struct grmkm_scm_job {
    uint32_t struct_size;  /* = sizeof(grmkm_scm_job) */
    uint32_t model_type;   /* GRMKM_SCM_CONJUNCTION / GRMKM_SCM_DISJUNCTION */
    uint32_t max_rules;    /* >= 1 */
    uint32_t tiebreak;     /* 1: risk tiebreaker (experiment_scm.py), 0: none */
    double p;              /* >= 0, finite */
    const uint64_t* pos;   /* P0: n_words words, genome g at bit 63 - g % 64 of word g / 64 */
    const uint64_t* neg;   /* N0: disjoint from P0 */
} grmkm_scm_job;

typedef struct grmkm_scm_step {
    uint64_t rule;             /* < 2U */
    double utility;            /* u* */
    uint32_t positive_errors;  /* e of the rule */
    uint32_t negative_covers;  /* c of the rule */
    uint64_t equiv_offset;     /* T of this step: equivalent[equiv_offset .. + equiv_count), ascending */
    uint64_t equiv_count;
} grmkm_scm_step;

/* Runs every fit to completion; the results stay in the context until the next run / build / load / reset.  Refuses
 * (GRMKM_E_UNSUPPORTED) a result that is one owner's slice of a multi-GPU merge. */
int grmkm_scm_run(grmkm_ctx* ctx, uint32_t n_fits, const grmkm_scm_job* jobs, const uint64_t* blacklist,
                  uint64_t n_blacklist);
/* Steps and equivalent rules of fit `fit`.  *n_steps / *n_equivalent receive the sizes; NULL or short buffers:
 * GRMKM_E_CAPACITY (sizes still written). */
int grmkm_scm_result(grmkm_ctx* ctx, uint32_t fit, grmkm_scm_step* steps, uint64_t steps_cap, uint64_t* n_steps,
                     uint64_t* equivalent, uint64_t equiv_cap, uint64_t* n_equivalent);

/*
 * CART decision trees (kover learning/learners/cart.py, gini criterion) on the resident matrix, many trees at once.
 * A node splits on k-mer j < U: the examples holding it go to the present child, the others to the absent child (rule
 * U + j is the same split, so only j < U is considered; a blacklist entry j or U + j removes k-mer j).  For a child
 * with a positive and b negative examples, A = w_pos * a, B = w_neg * b, S = A + B, term = (A * B) / S, each a
 * correctly rounded double operation in this order; score = term_present + term_absent (half the weighted Gini
 * impurity sum).  Admissible: both children non-empty, k-mer not blacklisted.  s* = min score over admissible splits,
 * T = {admissible j : score == s*}, the node's rule is min T.  A node is a leaf when depth == max_depth (root: 0),
 * a + b < min_samples_split, a == 0 or b == 0, or T is empty.  prediction = 1 iff A > B of the node's own counts.
 * Nodes are numbered breadth-first: level by level, in their parents' order, the present child before the absent
 * child; the root is 0.  Every level of all trees is one pass over the matrix on the device; only the best scores,
 * the tie list and the chosen rules' counts cross PCIe.
 */
typedef struct grmkm_cart_job {
    uint32_t struct_size;        /* = sizeof(grmkm_cart_job) */
    uint32_t max_depth;          /* >= 1 */
    uint32_t min_samples_split;  /* >= 2 */
    uint32_t reserved;           /* 0 */
    uint64_t equiv_cap;          /* per node, at most this many (the smallest) members of T are recorded */
    double w_neg;                /* class importance of the negatives: finite, > 0, <= 1e100 (no product overflows) */
    double w_pos;                /* the same for the positives */
    const uint64_t* pos;         /* n_words words, genome g at bit 63 - g % 64 of word g / 64 */
    const uint64_t* neg;         /* disjoint from pos */
} grmkm_cart_job;

typedef struct grmkm_cart_node {
    uint64_t rule;               /* k-mer index of the split (< U), UINT64_MAX: leaf */
    double score;                /* s* of the split; leaf: 0 */
    uint32_t depth;              /* root: 0 */
    uint32_t n_pos;              /* a: positive examples of the node */
    uint32_t n_neg;              /* b: negative examples of the node */
    uint32_t present_child;      /* node index, UINT32_MAX: leaf */
    uint32_t absent_child;
    uint32_t prediction;         /* 1 iff w_pos * a > w_neg * b (the leaf's output) */
    uint64_t equiv_offset;       /* the recorded members of T: equivalent[equiv_offset .. + equiv_count), ascending */
    uint64_t equiv_count;        /* min(|T|, equiv_cap) */
    uint64_t equiv_total;        /* |T| */
} grmkm_cart_node;

/* Grows every tree to completion; the results stay in the context until the next run / build / load / reset.  Refuses
 * (GRMKM_E_UNSUPPORTED) a result that is one owner's slice of a multi-GPU merge. */
int grmkm_cart_run(grmkm_ctx* ctx, uint32_t n_trees, const grmkm_cart_job* jobs, const uint64_t* blacklist,
                   uint64_t n_blacklist);
/* Nodes and equivalent rules of tree `tree`.  *n_nodes / *n_equivalent receive the sizes; NULL or short buffers:
 * GRMKM_E_CAPACITY (sizes still written). */
int grmkm_cart_result(grmkm_ctx* ctx, uint32_t tree, grmkm_cart_node* nodes, uint64_t nodes_cap, uint64_t* n_nodes,
                      uint64_t* equivalent, uint64_t equiv_cap, uint64_t* n_equivalent);

/*
 * Query: which genome rows of the inputs hold which k-mers, without building their matrix (a fitted model applied to
 * new genomes: its rules' k-mers; a marker panel: the k-mers of known genes).
 *
 * kmers[i] is packed as grmkm_copy_kmers_packed returns it (A0 C1 T2 G3, first base most significant, < 4^k), on
 * either strand; duplicates are allowed.  Column i of the answer is about canonical(kmers[i]) = min(forward, reverse
 * complement), the complement of code c being c ^ 2.  Genome g has column i set iff, among the valid k-mer windows of
 * g's inputs (the windows, records and FASTA/FASTQ rules of a build), at least min_abundance have the canonical k-mer
 * canonical(kmers[i]): the per-genome solid set before the singleton filter, so keep_singletons plays no part.  For a
 * k-mer that is a column of a build of the same inputs, the query column equals the matrix column bit for bit; every
 * other k-mer gives zeros, except a k-mer of exactly one genome when the build drops singletons.
 *
 * dst: row-major ceil(G/64) x n_kmers words, genome g at bit 63 - g % 64 of word row g / 64 (the matrix's layout), G
 * the genome count a build of these inputs would have (max row + 1, or grmkm_set_genome_count).
 *
 * The call reads the inputs added since the last reset, as grmkm_build does, and keeps them: a build or another query
 * can follow.  It changes nothing else in the context: the resident result, grmkm_get_stats, grmkm_stage_times and the
 * SCM and CART results stay as they are (grmkm_stats.device_bytes is the memory the context holds at the time of the
 * call, and counts the buffers a query keeps for the next one).  Rejected before any device work: a k-mer >= 4^k and a bad
 * stats->struct_size (GRMKM_E_INVALID), a GRMKM_FLAG_COUNTS context (GRMKM_E_INVALID: pooled counts have no genome
 * rows), cap < ceil(G/64) * n_kmers (GRMKM_E_CAPACITY).  n_kmers = 0 or G = 0 is valid and writes nothing.
 */
typedef struct grmkm_query_stats {
    uint32_t struct_size;     /* = sizeof(grmkm_query_stats) */
    uint32_t n_jobs;          /* row ranges the call was split into (each a pass over its rows' inputs) */
    uint64_t n_queries;       /* distinct canonical k-mers in the query */
    uint64_t n_bases, n_windows, n_records, n_input_bytes;   /* as grmkm_stats, for the queried inputs */
    uint64_t n_hits;          /* valid windows whose canonical k-mer is in the set */
    float ms;                 /* device time of the call, CUDA events */
} grmkm_query_stats;

int grmkm_query(grmkm_ctx* ctx, const uint64_t* kmers, uint64_t n_kmers, uint64_t* dst, uint64_t cap,
                grmkm_query_stats* stats /* may be NULL */);

/*
 * Evaluation: fitted models scored on example sets of the resident matrix, many at once (the held-out side of
 * cross-validation).  A job is one model and a pair of disjoint example masks pos / neg (n_words words, genome g at
 * bit 63 - g % 64 of word g / 64).  Only counts come back, as uint32 pairs, job after job in the order of the jobs:
 *
 *   GRMKM_EVAL_SCM   items = R rule indices < 2U, the model's own rules (a disjunction's absence twins already
 *                    applied: SetCoveringMachine.rule_indices).  R + 1 pairs (fn_r, fp_r), r = 0..R: fn_r = #pos the
 *                    model of the first r rules outputs 0 on, fp_r = #neg it outputs 1 on.  A conjunction outputs 1
 *                    iff all its rules do, a disjunction iff any does; the empty prefix outputs 1 / 0.
 *   GRMKM_EVAL_CART  items = n >= 1 nodes (root 0).  n pairs (p_i, q_i): the pos / neg examples that reach node i.
 *                    An example at split node i goes to present_child iff its bit in column kmer is set; a leaf
 *                    (kmer = UINT64_MAX) ends its walk, and its children are not read.
 *
 * Rejected before any device work (GRMKM_E_INVALID): a bad struct_size or kind, reserved != 0, an SCM rule >= 2U, a
 * CART job without nodes, a split k-mer >= U, a child index not greater than its parent's or >= n, a node with two
 * parents, overlapping masks, mask bits at rows >= n_genomes.  cap (in uint32 elements) below 2 x the pairs of all
 * jobs: GRMKM_E_CAPACITY.  A result that is one owner's slice of a multi-GPU merge: GRMKM_E_UNSUPPORTED.  One launch
 * (one warp per job) and one device->host copy of the counts; the context's SCM and CART results are left as they are.
 */
enum { GRMKM_EVAL_SCM = 0, GRMKM_EVAL_CART = 1 };

typedef struct grmkm_eval_node {
    uint64_t kmer;               /* split k-mer (< U), UINT64_MAX: leaf */
    uint32_t present_child;      /* node index (> this node's), read for a split node only */
    uint32_t absent_child;
} grmkm_eval_node;

typedef struct grmkm_eval_job {
    uint32_t struct_size;        /* = sizeof(grmkm_eval_job) */
    uint32_t kind;               /* GRMKM_EVAL_SCM / GRMKM_EVAL_CART */
    uint32_t model_type;         /* SCM: GRMKM_SCM_CONJUNCTION / GRMKM_SCM_DISJUNCTION; CART: 0 */
    uint32_t reserved;           /* 0 */
    uint64_t n_items;            /* SCM: R rules (0 allowed); CART: n nodes (>= 1) */
    const uint64_t* rules;       /* SCM: R rule indices */
    const grmkm_eval_node* nodes; /* CART: n nodes */
    const uint64_t* pos;         /* n_words words */
    const uint64_t* neg;         /* disjoint from pos */
} grmkm_eval_job;

int grmkm_eval_run(grmkm_ctx* ctx, uint32_t n_jobs, const grmkm_eval_job* jobs, uint32_t* counts, uint64_t cap);

/*
 * Sharded runs: learning and evaluation on the column slices of a multi-GPU build, the matrix never gathered.
 *
 * Rank r of P holds the global columns [col_offset, col_offset + U_r) of a matrix of n_kmers_total columns; the
 * slices, in rank order, tile [0, n_kmers_total) (the owner slices of grmkm_merge_partials do; so do column ranges
 * loaded with grmkm_load_result).  Every rank calls the same sharded function with the same jobs, blacklist and
 * n_kmers_total, and gets the same global result, bit for bit the result of the unsharded call on the whole matrix:
 * rule, k-mer, blacklist and split indices are global (presence rule j, absence rule n_kmers_total + j), and results
 * are read with grmkm_scm_result / grmkm_cart_result / the counts buffer as usual.
 *
 * The ranks talk through one collective, an all-gather of variable-size byte blocks: exchange(user, send, n, &recv,
 * sizes) returns in recv the concatenation of every rank's block in rank order (sizes[r] bytes from rank r), valid
 * until the next call on this rank.  A non-zero return aborts the run on this rank with GRMKM_E_INVALID.  The first
 * exchange of a run carries every rank's validation status, column range and n_kmers_total: if any rank fails (bad
 * jobs, no result, ranges that do not tile [0, n_kmers_total), ranks given different n_kmers_total), every rank
 * returns the first failing rank's code before any device work, and no rank is left waiting.  A rank that owns no
 * columns launches nothing but takes part in every exchange.
 *
 * Failures that are not collective: a bad shard (NULL, wrong struct_size, NULL exchange, rank >= n_ranks) returns on
 * that rank before the first exchange, and an error after it (device memory, a CUDA error, a failed exchange) returns
 * on the rank that meets it.  Either way the other ranks wait in their next exchange until it fails: the exchange
 * must give up after a timeout (distributed.ThreadExchange has one; a torch.distributed process group has its own), and
 * the caller treats such a failure on any rank as the failure of the whole run.
 * Per SCM step: the best keys (8 bytes per pending fit), the tie lists with their statistics, the chosen columns
 * (8 x n_words bytes each); per CART level: the best keys, the tie totals and lists, the split columns; per eval call:
 * the columns of the jobs' rules and split k-mers.
 */
typedef int (*grmkm_exchange_fn)(void* user, const void* send, uint64_t n, const void** recv, uint64_t* sizes /*[n_ranks]*/);

typedef struct grmkm_shard {
    uint32_t struct_size;        /* = sizeof(grmkm_shard) */
    uint32_t rank;               /* < n_ranks */
    uint32_t n_ranks;            /* >= 1 */
    uint32_t reserved;           /* 0 */
    uint64_t col_offset;         /* the global index of this slice's first column */
    uint64_t n_kmers_total;      /* U of the whole matrix */
    grmkm_exchange_fn exchange;  /* not NULL */
    void* user;                  /* passed to exchange */
} grmkm_shard;

int grmkm_scm_run_sharded(grmkm_ctx* ctx, uint32_t n_fits, const grmkm_scm_job* jobs, const uint64_t* blacklist,
                          uint64_t n_blacklist, const grmkm_shard* shard);
int grmkm_cart_run_sharded(grmkm_ctx* ctx, uint32_t n_trees, const grmkm_cart_job* jobs, const uint64_t* blacklist,
                           uint64_t n_blacklist, const grmkm_shard* shard);
int grmkm_eval_run_sharded(grmkm_ctx* ctx, uint32_t n_jobs, const grmkm_eval_job* jobs, uint32_t* counts, uint64_t cap,
                           const grmkm_shard* shard);

/* The words of columns idx[0 .. n) of the resident result, dst[w * n + i] = word row w of column idx[i] (n_words x n,
 * row-major), packed on the device: the columns a model needs without copying the whole matrix.  idx[i] >= n_kmers or
 * n >= 2^32: GRMKM_E_INVALID; cap < n_words x n: GRMKM_E_CAPACITY. */
int grmkm_copy_columns(grmkm_ctx* ctx, const uint64_t* idx, uint64_t n, uint64_t* dst, uint64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* GRMKM_H */
