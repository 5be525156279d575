"""Cross-validated selection on the resident matrix: wall time of a whole cross_validate_scm (5 folds, 2 model types,
10 p, up to 10 rules) and cross_validate_cart (5 folds + the full set, depths 1..10 x min samples {2, 5, 10}), the share
of their one eval_run, the host composition one can write without it (``predict`` per fit on its held-out rows, the
first ``get_columns`` copying the whole matrix to the host), and bit-exact checks.  Prints one JSON line (commit it
under profiles/).

Workloads and labels are tools/scm_bench.py's: synthetic 5 Mbp genomes built on the GPU -- C2's shape (100 genomes,
k = 31, singletons kept, W = 2) and 500 genomes (singletons dropped, W = 8).  A seeded 20 % of the genomes is the test
set, the rest the training set.

    python tools/selection_bench.py [--out FILE] [--repeats 3]
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

from scm_bench import P_GRID, WORKLOADS, build, card, labels_for  # noqa: E402

TYPES = ["conjunction", "disjunction"]
DEPTHS = list(range(1, 11))
MSS = [2, 5, 10]
FOLDS, MAX_RULES = 5, 10


def wall(fn, repeats):
    """Median wall time of repeated calls (each ends in a device synchronise) after one warm-up call, and the last result."""
    res = fn()
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        res = fn()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), res


def host_scm(rc, pos, neg, ids):
    """The composition a user writes today: fit_many, then predict of every prefix of every fold's machine."""
    from grm_b200.scm import SetCoveringMachine, fit_many
    k = FOLDS
    sets = [(ids[:len(pos)] == f, ids[len(pos):] == f) for f in range(k)]
    machines = [[SetCoveringMachine(t, p, MAX_RULES) for t in TYPES for p in P_GRID] for _ in range(k)]
    fit_many(rc, [(m, pos[~a], neg[~b]) for ms, (a, b) in zip(machines, sets) for m in ms])
    t0 = time.perf_counter()
    errors = np.zeros((len(TYPES), len(P_GRID), MAX_RULES), dtype=np.int64)
    for f, (a, b) in enumerate(sets):
        held = np.concatenate([pos[a], neg[b]])
        for c, m in enumerate(machines[f]):
            for r in range(1, MAX_RULES + 1):
                cut = SetCoveringMachine(m.model_type, m.p, r)
                cut.rule_indices = m.rule_indices[:r]
                pred = cut.predict(rc, held)
                errors[c // len(P_GRID), c % len(P_GRID), r - 1] += int((pred[:a.sum()] == 0).sum() + (pred[a.sum():] == 1).sum())
    return time.perf_counter() - t0, errors


def host_cart(rc, pos, neg, ids):
    """fit_many of the fold trees, then predict of every (depth, min samples) truncation on the held-out rows."""
    from grm_b200 import cart
    from grm_b200.model_selection import _truncate
    sets = [(ids[:len(pos)] == f, ids[len(pos):] == f) for f in range(FOLDS)]
    trees = [cart.DecisionTreeClassifier(max_depth=max(DEPTHS), min_samples_split=min(MSS)) for _ in sets]
    cart.fit_many(rc, [(t, pos[~a], neg[~b]) for t, (a, b) in zip(trees, sets)])
    t0 = time.perf_counter()
    errors = np.zeros((1, len(DEPTHS), len(MSS)), dtype=np.int64)
    for t, (a, b) in zip(trees, sets):
        held = np.concatenate([pos[a], neg[b]])
        for di, d in enumerate(DEPTHS):
            for si, s in enumerate(MSS):
                pred = _truncate(t, d, s).predict(rc, held)
                errors[0, di, si] += int((pred[:a.sum()] == 0).sum() + (pred[a.sum():] == 1).sum())
    return time.perf_counter() - t0, errors


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    import torch
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.learning import KmerRuleClassifications
    from grm_b200.model_selection import cross_validate_cart, cross_validate_scm
    from grm_b200.scm import SetCoveringMachine
    res = {"tool": "tools/selection_bench.py", "card": card(), "folds": FOLDS, "model_types": TYPES, "p_grid": P_GRID,
           "max_rules": MAX_RULES, "max_depths": DEPTHS, "min_samples_splits": MSS, "workloads": []}
    for name, G, keep in WORKLOADS:
        rng = np.random.default_rng(G)
        b = build(G, keep)
        U, W, _ = b.dims
        marker, labels = labels_for(b, G, rng)
        order = np.random.default_rng(G + 1).permutation(G)
        test, train = order[:G // 5], order[G // 5:]
        pos, neg = train[labels[train] == 1], train[labels[train] == 0]
        tpos, tneg = test[labels[test] == 1], test[labels[test] == 0]
        w = {"name": name, "genomes": G, "n_kmers": U, "n_words": W, "matrix_bytes": 8 * W * U, "marker_column": marker,
             "train": len(train), "test": len(test)}
        rc = KmerRuleClassifications(b, G)

        s_wall, s = wall(lambda: cross_validate_scm(rc, pos, neg, TYPES, P_GRID, MAX_RULES, FOLDS, test_pos=tpos,
                                                    test_neg=tneg), args.repeats)
        fits = (FOLDS + 1) * len(TYPES) * len(P_GRID)
        w["scm"] = {"wall_s": s_wall, "fit_s": s.seconds["fit"], "eval_s": s.seconds["eval"],
                    "eval_share": s.seconds["eval"] / s.seconds["total"], "fits": fits,
                    "eval_jobs": fits + len(TYPES) * len(P_GRID), "selected": s.selected, "test": s.test,
                    "note": "median wall of the whole call over the repeats; fit_s / eval_s: the last call's fit_many and eval_run"}
        c_wall, c = wall(lambda: cross_validate_cart(rc, pos, neg, [None], DEPTHS, MSS, FOLDS, test_pos=tpos,
                                                     test_neg=tneg), args.repeats)
        w["cart"] = {"wall_s": c_wall, "fit_s": c.seconds["fit"], "eval_s": c.seconds["eval"],
                     "eval_share": c.seconds["eval"] / c.seconds["total"], "trees": FOLDS + 1,
                     "nodes_full_tree": len(c.model.nodes), "selected": c.selected, "test": c.test}

        # the host compositions, each on a fresh KmerRuleClassifications: its first get_columns copies the whole matrix
        ids = s.fold_ids
        host_s, host_err = host_scm(KmerRuleClassifications(b, G), pos, neg, ids)
        host_c, host_cerr = host_cart(KmerRuleClassifications(b, G), pos, neg, ids)
        w["host_scm_predict_s"] = host_s
        w["host_cart_predict_s"] = host_c
        w["host_note"] = ("predict per (fold, candidate) on the held-out rows after the same batched fit; the first "
                          "get_columns copies the whole matrix to pageable host memory; fits not included")
        grid = np.array([g["cv_errors"] for g in s.grid]).reshape(MAX_RULES, len(TYPES), len(P_GRID)).transpose(1, 2, 0)
        t, p, r = TYPES.index(s.selected["model_type"]), P_GRID.index(s.selected["p"]), s.selected["max_rules"]
        fresh = SetCoveringMachine(TYPES[t], P_GRID[p], r).fit(rc, pos, neg)
        d, mss = c.selected["max_depth"], c.selected["min_samples_split"]
        direct = DecisionTreeClassifier(max_depth=d, min_samples_split=mss).fit(rc, pos, neg)
        same_tree = len(direct.nodes) == len(c.model.nodes) and all(
            (x.rule is None) == (y.rule is None) and (x.rule is None or x.rule == y.rule) and x[1:7] == y[1:7]
            and x.prediction == y.prediction and np.array_equal(x.equivalent_rules, y.equivalent_rules)
            for x, y in zip(direct.nodes, c.model.nodes))
        test_pred = direct.predict(rc, np.concatenate([tpos, tneg]))
        w["checks"] = {
            "scm_grid_equals_host_composition": "ok" if np.array_equal(grid, host_err) else "FAILED",
            "cart_grid_equals_host_composition": "ok" if [g["cv_errors"] for g in c.grid] == host_cerr.reshape(-1).tolist() else "FAILED",
            "scm_model_equals_fresh_fit": "ok" if fresh.rule_indices == s.model.rule_indices else "FAILED",
            "cart_model_equals_direct_fit": "ok" if same_tree else "FAILED",
            "cart_test_metrics_equal_predict": "ok" if (c.test["fn"], c.test["fp"]) == (
                int((test_pred[:len(tpos)] == 0).sum()), int((test_pred[len(tpos):] == 1).sum())) else "FAILED",
        }
        res["workloads"].append(w)
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
