"""Learning on the distinct presence patterns: U, P and the device time of grmkm_patterns, then the whole matrix against
a PatternRuleClassifications view, alternated in one process -- fit_many of the 120-fit SCM grid (10 rules) and of 6
CART trees (depth 10), cross_validate_scm and cross_validate_cart (the view's construction included) -- with a
bit-exact check of every view result against the whole-matrix one.  Prints one JSON line (commit it under profiles/).

Workloads and labels are tools/scm_bench.py's: synthetic 5 Mbp genomes built on the GPU -- C2's shape (100 genomes,
k = 31, singletons kept, W = 2) and 500 genomes (singletons dropped, W = 8).

    python tools/pattern_bench.py [--out FILE] [--repeats 3]
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

from scm_bench import P_GRID, WORKLOADS, build, card, grid_jobs, labels_for  # noqa: E402

TYPES = ["conjunction", "disjunction"]
MAX_RULES, DEPTH, FOLDS = 10, 10, 5


def alternate(fns, repeats):
    """Median wall time of each fn (calls that end in a device synchronise), the fns alternated, after one warm-up
    round; and the last results."""
    res = [fn() for fn in fns]
    times = [[] for _ in fns]
    for _ in range(repeats):
        for i, fn in enumerate(fns):
            t0 = time.perf_counter()
            res[i] = fn()
            times[i].append(time.perf_counter() - t0)
    return [float(np.median(t)) for t in times], res


def scm_models(ms):
    return [(m.rule_indices, [(it.rule, np.float64(it.utility).view(np.int64), it.positive_errors, it.negative_covers,
                               it.equivalent_rules.tolist()) for it in m.iterations]) for m in ms]


def selection_json(res):
    d = res.to_dict()
    d.pop("seconds")
    return json.dumps(d, sort_keys=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    import torch
    from grm_b200 import cart, scm
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.learning import KmerRuleClassifications, PatternRuleClassifications
    from grm_b200.model_selection import cross_validate_cart, cross_validate_scm
    res = {"tool": "tools/pattern_bench.py", "card": card(), "scm_fits": 120, "scm_max_rules": MAX_RULES,
           "cart_trees": FOLDS + 1, "cart_max_depth": DEPTH, "repeats": args.repeats, "workloads": []}
    for name, G, keep in WORKLOADS:
        rng = np.random.default_rng(G)
        b = build(G, keep)
        U, W, _ = b.dims
        marker, labels = labels_for(b, G, rng)
        w = {"name": name, "genomes": G, "n_kmers": U, "n_words": W}
        with KmerMatrixBuilder(k=31) as dst:
            b.patterns(dst)                                       # warm-up
            ms = []
            for _ in range(max(3, args.repeats)):
                _, _, _, st = b.patterns(dst, with_stats=True)
                ms.append(st["ms"])
        w.update(n_patterns=st["n_patterns"], u_over_p=U / max(1, st["n_patterns"]), rounds=st["n_rounds"],
                 patterns_ms=float(np.median(ms)), patterns_note="device time of grmkm_patterns (CUDA events), median")
        rc = KmerRuleClassifications(b, G)
        view = PatternRuleClassifications(rc)

        jobs = grid_jobs(labels, W, np.random.default_rng(G + 2), MAX_RULES)

        def scm_fit(r):
            ms_ = [scm.SetCoveringMachine(TYPES[mt], p, MAX_RULES) for _, _, _, p, mt in jobs]
            scm.fit_many(r, [(m, pos, neg) for m, (_, pos, neg, _, _) in zip(ms_, jobs)])
            return scm_models(ms_)

        folds = [(pos, neg) for _, pos, neg, p, mt in jobs if p == P_GRID[0] and mt == 0]

        def cart_fit(r):
            ts = [cart.DecisionTreeClassifier(max_depth=DEPTH) for _ in folds]
            cart.fit_many(r, [(t, pos, neg) for t, (pos, neg) in zip(ts, folds)])
            return [str(t.nodes) for t in ts]

        pos, neg = np.nonzero(labels == 1)[0], np.nonzero(labels == 0)[0]

        def cv_scm(r, make_view):
            if make_view:
                r = PatternRuleClassifications(r)
            out = selection_json(cross_validate_scm(r, pos, neg, TYPES, P_GRID, MAX_RULES, FOLDS))
            if make_view:
                r.close()
            return out

        def cv_cart(r, make_view):
            if make_view:
                r = PatternRuleClassifications(r)
            out = selection_json(cross_validate_cart(r, pos, neg, [None], list(range(1, DEPTH + 1)), [2, 5, 10], FOLDS))
            if make_view:
                r.close()
            return out

        checks = {}
        for key, fns in (("scm_fit_many_120", (lambda: scm_fit(rc), lambda: scm_fit(view))),
                         ("cart_fit_many_6", (lambda: cart_fit(rc), lambda: cart_fit(view))),
                         ("cross_validate_scm", (lambda: cv_scm(rc, False), lambda: cv_scm(rc, True))),
                         ("cross_validate_cart", (lambda: cv_cart(rc, False), lambda: cv_cart(rc, True)))):
            (t_whole, t_view), (r_whole, r_view) = alternate(fns, args.repeats)
            w[key] = {"whole_s": t_whole, "view_s": t_view, "speedup": t_whole / t_view}
            checks[key + "_equal"] = "ok" if r_whole == r_view else "FAILED"
        w["timing_note"] = ("median wall time over the repeats, whole matrix and view alternated; each call ends in a "
                            "device synchronise; the cross_validate view times include building the view")
        w["checks"] = checks
        res["workloads"].append(w)
        view.close()
        b.close()
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if any(v != "ok" for w in res["workloads"] for v in w["checks"].values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
