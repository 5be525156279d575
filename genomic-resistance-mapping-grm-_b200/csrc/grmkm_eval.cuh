// grmkm_eval.cuh -- fitted models scored on example sets of the resident matrix (the held-out side of Kover's
// cross-validation, `kover learn scm|tree --hp-choice cv`).  A batch of evaluation jobs is one launch: one warp per job,
// and only counts are written.
//
//   SCM job   lanes hold consecutive words of the examples; o = the output word-mask of the prefix of r rules (all ones
//             for an empty conjunction, zeros for an empty disjunction), one column gathered per rule (matrix-pitch
//             access, inverted for an absence rule U + j) and folded in with & (conjunction) or | (disjunction).  Per
//             prefix: fn = popc(pos & ~o), fp = popc(neg & o), warp-reduced with redux.sync.
//   CART job  lanes hold consecutive examples; each walks the tree from the root, one bit of the split column per level
//             (the warp's 32 examples share a word, so the load is a broadcast), and every node it visits counts it.
//             Lanes at the same node add once per warp (match.any).  No example mask is kept per node: the walk needs
//             no scratch whatever the tree's size, and takes any node order in which a child follows its parent.
//
// counts: uint32 pairs, job after job from args[i].out.  W > 32 (SCM) adds per 32-word chunk and a CART node is counted
// by several warps' walks, so counts are accumulated with atomicAdd into a zeroed buffer (integer sums: the order does
// not matter).
#pragma once
#include <cstdint>

namespace grmkm {

constexpr uint32_t kEvalThreads = 256;
constexpr uint32_t kEvalLeaf = 0xFFFFFFFFu;     // no node: the walk has passed a leaf

enum : uint32_t { EVAL_SCM = 0, EVAL_CART = 1 };

struct EvalJobArg {
    uint32_t kind;                // EVAL_SCM / EVAL_CART
    uint32_t conjunction;         // SCM: 1 conjunction, 0 disjunction
    uint32_t n;                   // SCM: rules; CART: nodes
    uint32_t pad;
    unsigned long long items;     // offset of the job's rules / nodes
    unsigned long long out;       // offset of the job's first count pair
};

// = grmkm_eval_node
struct EvalNode {
    unsigned long long kmer;      // split column, UINT64_MAX: leaf
    uint32_t present, absent;     // children (read for a split node only)
};

__device__ __forceinline__ void eval_scm(const EvalJobArg& a, const unsigned long long* __restrict__ matrix,
                                         unsigned long long U, unsigned long long pitch, uint32_t W,
                                         const unsigned long long* __restrict__ rules, const unsigned long long* P,
                                         const unsigned long long* N, uint32_t* __restrict__ cnt, uint32_t lane) {
    for (uint32_t w0 = 0; w0 < W; w0 += 32) {
        const uint32_t w = w0 + lane;
        const bool ok = w < W;
        const unsigned long long p = ok ? P[w] : 0ULL, q = ok ? N[w] : 0ULL;
        unsigned long long o = a.conjunction ? ~0ULL : 0ULL;
        for (uint32_t r = 0;; ++r) {
            const uint32_t fn = __reduce_add_sync(0xffffffffu, (uint32_t)__popcll(p & ~o));
            const uint32_t fp = __reduce_add_sync(0xffffffffu, (uint32_t)__popcll(q & o));
            if (lane == 0) {
                if (fn) atomicAdd(cnt + 2 * (a.out + r), fn);
                if (fp) atomicAdd(cnt + 2 * (a.out + r) + 1, fp);
            }
            if (r == a.n) break;
            const unsigned long long rule = rules[a.items + r];
            const bool absent = rule >= U;
            unsigned long long x = ok ? __ldg(matrix + (unsigned long long)w * pitch + (absent ? rule - U : rule)) : 0ULL;
            if (absent) x = ~x;
            o = a.conjunction ? (o & x) : (o | x);
        }
    }
}

__device__ __forceinline__ void eval_cart(const EvalJobArg& a, const unsigned long long* __restrict__ matrix,
                                          unsigned long long pitch, uint32_t W, const EvalNode* __restrict__ nodes,
                                          const unsigned long long* P, const unsigned long long* N,
                                          uint32_t* __restrict__ cnt, uint32_t lane) {
    const EvalNode* nd = nodes + a.items;
    for (uint32_t g0 = 0; g0 < 64 * W; g0 += 32) {
        const uint32_t wi = g0 >> 6, sh = 63u - ((g0 + lane) & 63u);
        const bool is_p = (P[wi] >> sh) & 1ULL, is_n = (N[wi] >> sh) & 1ULL;
        const uint32_t pm = __ballot_sync(0xffffffffu, is_p), nm = __ballot_sync(0xffffffffu, is_n);
        if (!(pm | nm)) continue;
        uint32_t node = (is_p || is_n) ? 0u : kEvalLeaf;
        for (;;) {
            const bool act = node != kEvalLeaf;
            const uint32_t am = __ballot_sync(0xffffffffu, act);
            if (!am) break;
            if (act) {
                const uint32_t grp = __match_any_sync(am, node);
                if (lane == (uint32_t)__ffs(grp) - 1) {
                    const uint32_t cp = __popc(grp & pm), cn = __popc(grp & nm);
                    if (cp) atomicAdd(cnt + 2 * (a.out + node), cp);
                    if (cn) atomicAdd(cnt + 2 * (a.out + node) + 1, cn);
                }
                const EvalNode e = nd[node];
                if (e.kmer == ~0ULL) {
                    node = kEvalLeaf;
                } else {
                    const unsigned long long x = __ldg(matrix + (unsigned long long)wi * pitch + e.kmer);
                    node = ((x >> sh) & 1ULL) ? e.present : e.absent;
                }
            }
        }
    }
}

// warp i of the grid takes jobs i, i + warps, ...; masks[job][0..1][W] = pos, neg
__global__ void __launch_bounds__(kEvalThreads)
k_eval(const unsigned long long* __restrict__ matrix, unsigned long long U, unsigned long long pitch, uint32_t W,
       const EvalJobArg* __restrict__ args, uint32_t n_jobs, const unsigned long long* __restrict__ rules,
       const EvalNode* __restrict__ nodes, const unsigned long long* __restrict__ masks, uint32_t* __restrict__ cnt) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = gridDim.x * (kEvalThreads / 32);
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n_jobs; i += warps) {
        const EvalJobArg a = args[i];
        const unsigned long long* P = masks + (size_t)i * 2 * W;
        if (a.kind == EVAL_SCM) eval_scm(a, matrix, U, pitch, W, rules, P, P + W, cnt, lane);
        else eval_cart(a, matrix, pitch, W, nodes, P, P + W, cnt, lane);
    }
}

}  // namespace grmkm
