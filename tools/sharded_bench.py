"""Learning on column slices: the whole-matrix grmkm_scm_run / grmkm_cart_run against the same runs on P = 2 / 4 / 8
column slices of the matrix, each in its own context on this GPU, driven by P threads through a ThreadExchange.  The
difference is the cost of the exchanges, the host merges and the split launches (the slices share one GPU here, so
the scans are not faster; across GPUs each slice's scan would be about 1/P of the whole).  Bit-exact checks of every
sharded result against the whole.  Prints one JSON line (commit it under profiles/).

Workloads: the two matrices of tools/scm_bench.py (C2's shape, 100 genomes, and 500 genomes).  SCM: the 120-fit
CV x p x model-type grid with 10 rules.  CART: 12 trees (6 fold sets x 2 class weightings), max_depth 5, 100 recorded
equivalent rules per node.  Host clock around each call (every call ends in a device synchronise on every rank), at
least 10 calls and min-seconds per row; the median and the spread (min, max) are reported.

    python tools/sharded_bench.py [--out FILE] [--min-seconds 3.0]
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from scm_bench import WORKLOADS, build, card, grid_jobs, labels_for, mask  # noqa: E402

RANKS = [2, 4, 8]


def timed(fn, min_seconds):
    """Per-call host times (ms) over at least min_seconds and 10 calls, after two warm-up calls: median and spread."""
    fn()
    fn()
    ts, t0 = [], time.perf_counter()
    while time.perf_counter() - t0 < min_seconds or len(ts) < 10:
        t = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t) * 1e3)
    return {"median": round(float(np.median(ts)), 3), "min": round(min(ts), 3), "max": round(max(ts), 3), "calls": len(ts)}


def run_row(ranks, scm, cart, steps, levels):
    return {"ranks": ranks, "scm_ms": scm, "scm_ms_per_step_median": round(scm["median"] / steps, 4),
            "cart_ms": cart, "cart_ms_per_level_median": round(cart["median"] / levels, 4)}


def slices(kmers, matrix, G, P):
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import ThreadExchange
    from grm_b200.learning import ShardedRuleClassifications
    U = len(kmers)
    cuts = [U * r // P for r in range(P + 1)]
    ex = ThreadExchange.group(P, timeout=300)
    rcs = []
    for r in range(P):
        b = KmerMatrixBuilder(k=31)
        b.load_result(kmers[cuts[r]:cuts[r + 1]], np.ascontiguousarray(matrix[:, cuts[r]:cuts[r + 1]]), G)
        rcs.append(ShardedRuleClassifications(b, G, r, P, [cuts[q + 1] - cuts[q] for q in range(P)], ex[r]))
    return rcs


def on_all(rcs, fn):
    out = [None] * len(rcs)

    def work(r):
        out[r] = fn(rcs[r])

    threads = [threading.Thread(target=work, args=(r,)) for r in range(len(rcs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if any(o is None for o in out):
        raise RuntimeError("a rank failed")
    return out


def same(a, b):
    return len(a) == len(b) and all(x[0].tobytes() == y[0].tobytes() and np.array_equal(x[1], y[1]) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=3.0)
    args = ap.parse_args()
    res = {"tool": "tools/sharded_bench.py", "card": card(), "workloads": [],
           "torchrun": "not measured (one GPU): the multi-process route and gather() + load_result + fit"}
    for name, G, keep in WORKLOADS:
        rng = np.random.default_rng(G)
        b = build(G, keep)
        U, W, _ = b.dims
        _, labels = labels_for(b, G, rng)
        sjobs = [j for j, *_ in grid_jobs(labels, W, rng, 10)]
        fold = rng.permutation(G) % 5
        cjobs = []
        for f in list(range(5)) + [None]:
            train = np.ones(G, dtype=bool) if f is None else fold != f
            pos, neg = np.nonzero(train & (labels == 1))[0], np.nonzero(train & (labels == 0))[0]
            for w in ((1.0, 1.0), (0.5, 2.0)):
                cjobs.append((5, 2, 100, w[0], w[1], mask(pos, W), mask(neg, W)))
        want_s, want_c = b.scm_run(sjobs), b.cart_run(cjobs)
        steps = max(len(s) for s, _ in want_s)
        levels = 1 + max(int(n["depth"].max()) for n, _ in want_c)
        w = {"name": name, "genomes": G, "n_kmers": U, "n_words": W, "scm_fits": len(sjobs), "scm_steps": steps,
             "cart_trees": len(cjobs), "cart_levels": levels, "runs": []}
        w["runs"].append(run_row("whole", timed(lambda: b.scm_run(sjobs), args.min_seconds),
                                 timed(lambda: b.cart_run(cjobs), args.min_seconds), steps, levels))
        kmers, matrix = b.kmers(), b.matrix()
        b.close()
        for P in RANKS:
            rcs = slices(kmers, matrix, G, P)
            got_s = on_all(rcs, lambda rc: rc.builder.scm_run(sjobs, shard=rc))
            got_c = on_all(rcs, lambda rc: rc.builder.cart_run(cjobs, shard=rc))
            row = run_row(P, timed(lambda: on_all(rcs, lambda rc: rc.builder.scm_run(sjobs, shard=rc)), args.min_seconds),
                          timed(lambda: on_all(rcs, lambda rc: rc.builder.cart_run(cjobs, shard=rc)), args.min_seconds),
                          steps, levels)
            row["scm_bit_exact"] = all(same(g, want_s) for g in got_s)
            row["cart_bit_exact"] = all(same(g, want_c) for g in got_c)
            w["runs"].append(row)
            for rc in rcs:
                rc.builder.close()
        res["workloads"].append(w)
        print(json.dumps(w), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
