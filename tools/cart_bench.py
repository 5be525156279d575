"""CART on the resident matrix: ms per tree of grmkm_cart_run for one tree and for 6 trees batched (5 CV training folds
+ the full set), ms per level against the open nodes of that level (the marginal cost of a node at a level), the host
composition one can write without it (KmerRuleClassifications.sum_rows per class + numpy Gini, argmin and ties) for
the root node, and bit-exact checks.  Prints one JSON line (commit it under profiles/).

Workloads and labels are tools/scm_bench.py's: synthetic 5 Mbp genomes built on the GPU -- C2's shape (100 genomes,
k = 31, singletons kept, W = 2) and 500 genomes (singletons dropped, W = 8).  Both matrices exceed the 126 MB L2.

    python tools/cart_bench.py [--out FILE] [--min-seconds 0.5] [--max-depth 10] [--equiv-cap 100]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from scm_bench import COPY_PEAK_GBS, WORKLOADS, build, card, labels_for, mask, timed  # noqa: E402


def fold_sets(labels, rng):
    """(pos rows, neg rows) of the 5 CV training folds and of the full set."""
    G = len(labels)
    fold = rng.permutation(G) % 5
    out = []
    for f in list(range(5)) + [None]:
        train = np.ones(G, dtype=bool) if f is None else fold != f
        out.append((np.nonzero(train & (labels == 1))[0], np.nonzero(train & (labels == 0))[0]))
    return out


def scanned_per_level(nodes, max_depth, min_samples_split):
    """Open nodes (scanned by the level's pass) per depth: every node no stop rule made a leaf before the scan."""
    n = nodes["n_pos"].astype(np.int64) + nodes["n_neg"]
    ok = (nodes["depth"] < max_depth) & (n >= min_samples_split) & (nodes["n_pos"] > 0) & (nodes["n_neg"] > 0)
    return np.bincount(nodes["depth"][ok], minlength=max_depth)[:max_depth]


def host_root(rc, pos, neg, U):
    """The root node written with what the package offered before grmkm_cart_run: sum_rows per class, numpy Gini."""
    sp = rc.sum_rows(pos)[:U].astype(np.int64)
    sn = rc.sum_rows(neg)[:U].astype(np.int64)
    a, b = len(pos), len(neg)

    def term(x, y):
        A, B = x.astype(np.float64), y.astype(np.float64)
        with np.errstate(invalid="ignore", divide="ignore"):
            return (A * B) / (A + B)

    score = term(sp, sn) + term(a - sp, b - sn)
    ok = (sp + sn > 0) & (a - sp + b - sn > 0)
    best = score[ok].min()
    T = np.nonzero(ok & (score == best))[0]
    return int(T[0]), float(best), len(T)


def same(x, y):
    return len(x) == len(y) and all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(x, y))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=0.5)
    ap.add_argument("--max-depth", type=int, default=10)
    ap.add_argument("--equiv-cap", type=int, default=100)
    args = ap.parse_args()
    import torch
    from grm_b200.learning import KmerRuleClassifications
    D, mss, cap = args.max_depth, 2, args.equiv_cap
    res = {"tool": "tools/cart_bench.py", "card": card(), "copy_peak_gbs": COPY_PEAK_GBS, "max_depth": D,
           "min_samples_split": mss, "equiv_cap": cap, "workloads": []}
    for name, G, keep in WORKLOADS:
        rng = np.random.default_rng(G)
        b = build(G, keep)
        U, W, _ = b.dims
        marker, labels = labels_for(b, G, rng)
        sets = fold_sets(labels, rng)
        w = {"name": name, "genomes": G, "k": 31, "keep_singletons": keep, "n_kmers": U, "n_words": W,
             "matrix_bytes": 8 * W * U, "marker_column": marker, "positives": int(labels.sum())}

        def jobs(depth, which):
            return [(depth, mss, cap, 1.0, 1.0, mask(p, W), mask(n, W)) for p, n in which]

        for label, which in (("one_tree", sets[-1:]), ("six_trees", sets)):
            J = {d: jobs(d, which) for d in range(1, D + 1)}           # masks built outside the timed calls
            trees = b.cart_run(J[D])
            open_per_level = sum(scanned_per_level(t, D, mss) for t, _ in trees)
            levels = int(np.nonzero(open_per_level)[0].max()) + 1
            # T(d) = one run with max_depth = d scans levels 0 .. d - 1 (a truncation of the same trees)
            t_d = {}
            for d in range(1, levels + 1):
                t_d[d], _ = timed(lambda: b.cart_run(J[d]), args.min_seconds)
            ms, n = timed(lambda: b.cart_run(J[D]), args.min_seconds)
            per_level = [{"level": l, "open_nodes": int(open_per_level[l]),
                          "ms": t_d[1] if l == 0 else t_d[l + 1] - t_d[l]} for l in range(levels)]
            x = np.array([p["open_nodes"] for p in per_level], dtype=np.float64)
            y = np.array([p["ms"] for p in per_level])
            slope, icpt = np.polyfit(x, y, 1) if len(x) > 1 and np.ptp(x) > 0 else (float("nan"), float("nan"))
            w[label] = {"trees": len(which), "ms_per_call": ms, "calls": n, "ms_per_tree": ms / len(which),
                        "nodes": [int(len(t)) for t, _ in trees], "levels": levels, "per_level": per_level,
                        "fit_ms_per_open_node_level": float(slope), "fit_ms_per_level_fixed": float(icpt),
                        "note": "ms per level = T(max_depth = l + 1) - T(max_depth = l), CUDA events around whole calls; "
                                "fit: least squares of ms per level against its open nodes"}
        batch = b.cart_run(jobs(D, sets))
        alone = [b.cart_run(jobs(D, [s]))[0] for s in sets]
        w["batched_equals_one_at_a_time"] = same(batch, alone)
        # the host composition for the root node only
        rc = KmerRuleClassifications(b, G)
        pos, neg = sets[-1]
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < max(args.min_seconds, 2.0) or n < 2:
            host = host_root(rc, pos, neg, U)
            n += 1
        host_ms = (time.perf_counter() - t0) * 1e3 / n
        root = alone[-1][0][0]
        scanned = int(scanned_per_level(alone[-1][0], D, mss).sum())
        w["host_root_ms"] = host_ms
        w["host_root_note"] = "KmerRuleClassifications.sum_rows per class (2 x U x 4 bytes to the host) + numpy Gini, argmin, ties"
        w["host_root_same_split"] = bool(host[0] == int(root["rule"]) and host[1] == float(root["score"])
                                         and host[2] == int(root["equiv_total"]))
        w["host_tree_ms_extrapolated"] = host_ms * scanned
        w["host_tree_note"] = f"extrapolation, not measured: host_root_ms x {scanned} scanned nodes of the full-set tree"
        res["workloads"].append(w)
        b.close()
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
