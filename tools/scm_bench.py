"""Set Covering Machine on the resident matrix: per-step time of grmkm_scm_run at F = 1 / 20 / 120 fits, the host
composition one can write without it (KmerRuleClassifications.sum_rows twice + numpy utilities, argmax and ties), the
whole CV x p x model-type grid, and bit-exact checks.  Prints one JSON line (commit it under profiles/).

Workloads: synthetic 5 Mbp genomes of synth.py built on the GPU -- C2's shape (100 genomes, k = 31, singletons kept,
W = 2) and 500 genomes (singletons dropped, W = 8: the row-block build path).  Both matrices exceed the 126 MB L2.
Labels are seeded: a planted marker column (present in 40-60 % of the genomes) XOR 10 % noise.

    python tools/scm_bench.py [--out FILE] [--min-seconds 1.0]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

P_GRID = [0.1, 0.178, 0.316, 0.562, 1.0, 1.778, 3.162, 5.623, 10.0, 999999.0]      # Kover's default hp grid
COPY_PEAK_GBS = 6552.0        # measured device-to-device copy on a B200 (BASELINE.md)
WORKLOADS = [("c2_100_genomes", 100, True), ("500_genomes_row_blocks", 500, False)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.strip().split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def build(G, keep):
    import torch
    from grm_b200 import synth
    from grm_b200.builder import KmerMatrixBuilder
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1)
    b = KmerMatrixBuilder(k=31, keep_singletons=keep)
    lay, total, spans = synth.build_layout(cfg, list(range(G)))
    buf = torch.empty(max(total, 16), dtype=torch.uint8, device="cuda")
    b._check(b._lib.grmkm_synth_fasta_device(b._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes, C.c_void_p(buf.data_ptr()), total))
    torch.cuda.synchronize()
    b.set_genome_count(G)
    b.add_genomes(np.arange(G, dtype=np.uint32), np.array([buf.data_ptr() + o for o, _ in spans], dtype=np.uint64),
                  np.array([n for _, n in spans], dtype=np.uint64), on_device=True)
    b.build()
    del buf
    return b


def labels_for(b, G, rng):
    U, W, _ = b.dims
    probe = rng.choice(U, size=min(U, 200_000), replace=False)
    sums = b.sum_rows(np.full(W, np.uint64(0xFFFFFFFFFFFFFFFF)))[probe]          # rows >= G are never set
    cand = probe[(sums >= 0.4 * G) & (sums <= 0.6 * G)]
    marker = int(rng.choice(cand))
    col = b.matrix()[:, marker]
    bits = np.array([(int(col[g // 64]) >> (63 - g % 64)) & 1 for g in range(G)], dtype=np.uint8)
    return marker, bits ^ (rng.random(G) < 0.1).astype(np.uint8)


def mask(rows, W):
    m = np.zeros(W, dtype=np.uint64)
    for g in rows:
        m[g // 64] |= np.uint64(1) << np.uint64(63 - g % 64)
    return m


def grid_jobs(labels, W, rng, max_rules):
    """10 p x 2 model types x (5 CV folds + the full training set) = 120 fits, as (job, pos rows, neg rows, p, type)."""
    G = len(labels)
    fold = rng.permutation(G) % 5
    out = []
    for f in list(range(5)) + [None]:
        train = np.ones(G, dtype=bool) if f is None else fold != f
        pos, neg = np.nonzero(train & (labels == 1))[0], np.nonzero(train & (labels == 0))[0]
        for mt in (0, 1):
            for p in P_GRID:
                out.append(((mt, p, max_rules, True, mask(pos, W), mask(neg, W)), pos, neg, p, mt))
    return out


def timed(fn, min_seconds):
    """CUDA events around repeated calls (each ends in a device synchronise) over at least min_seconds."""
    import torch
    fn()                                    # warm-up: modules, buffers, shapes
    fn()
    n, total = 0, 0.0
    while total < min_seconds * 1e3:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        n += 1
    return total / n, n


def host_step(rc, pos, neg, p, U):
    """One greedy step written with what the package offered before grmkm_scm_run (the reference's own loop)."""
    sp, sn = rc.sum_rows(pos), rc.sum_rows(neg)
    e = len(pos) - sp.astype(np.int64)
    c = len(neg) - sn.astype(np.int64)
    u = c.astype(np.float64) - p * e.astype(np.float64)
    best = u.max()
    T = np.nonzero((u == best) & ((c > 0) | (e > 0)))[0]
    return int(T.min()) if len(T) else -1


def same(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON line to this file")
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--oracle-fits", type=int, default=2, help="fits of the 100-genome grid checked against the numpy reference")
    args = ap.parse_args()
    import torch
    from grm_b200.learning import KmerRuleClassifications
    from tests.scm_oracle import scm_fit
    res = {"tool": "tools/scm_bench.py", "card": card(), "copy_peak_gbs": COPY_PEAK_GBS, "p_grid": P_GRID, "workloads": []}
    for name, G, keep in WORKLOADS:
        rng = np.random.default_rng(G)
        b = build(G, keep)
        U, W, _ = b.dims
        marker, labels = labels_for(b, G, rng)
        w = {"name": name, "genomes": G, "k": 31, "keep_singletons": keep, "n_kmers": U, "n_words": W, "rules": 2 * U,
             "matrix_bytes": 8 * W * U, "marker_column": marker, "positives": int(labels.sum()), "per_step": {}}
        jobs10 = grid_jobs(labels, W, rng, 10)
        full = [j for j in jobs10 if len(j[1]) + len(j[2]) == G]
        sets = {1: [full[4]], 20: full, 120: jobs10}           # F = 1: conjunction, p = 1, all examples
        assert len(sets[20]) == 20 and len(sets[120]) == 120
        for F, js in sets.items():
            one_step = [(mt, p, 1, tb, pm, nm) for (mt, p, _, tb, pm, nm), *_ in js]
            ms, n = timed(lambda: b.scm_run(one_step), args.min_seconds)
            w["per_step"][str(F)] = {"ms": ms, "calls": n, "gb_per_s": 8 * W * U / (ms * 1e-3) / 1e9,
                                     "frac_of_copy_peak": 8 * W * U / (ms * 1e-3) / 1e9 / COPY_PEAK_GBS,
                                     "popc64_per_s": 2.0 * F * W * U / (ms * 1e-3),
                                     "note": "one scm_run with max_rules = 1: upload of the masks + one greedy step of every fit"}
        # the host composition one can write without grmkm_scm_run, at F = 1
        rc = KmerRuleClassifications(b, G)
        (_, p1, _, _, _, _), pos1, neg1, _, _ = sets[1][0]
        t0, n = time.perf_counter(), 0
        while time.perf_counter() - t0 < max(args.min_seconds, 2.0) or n < 2:
            host_rule = host_step(rc, pos1, neg1, p1, U)
            n += 1
        w["host_step_f1_ms"] = (time.perf_counter() - t0) * 1e3 / n
        w["host_step_f1_note"] = "KmerRuleClassifications.sum_rows twice (2 x U x 4 bytes to the host) + numpy utilities, max, ties"
        mt1, _, _, _, pm1, nm1 = sets[1][0][0]
        gpu1 = b.scm_run([(mt1, p1, 1, False, pm1, nm1)])[0]
        w["host_step_same_rule"] = bool(len(gpu1[0]) and int(gpu1[0][0]["rule"]) == host_rule) if host_rule >= 0 else len(gpu1[0]) == 0
        # the whole grid: 120 fits x up to 10 rules
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        batch = b.scm_run([j[0] for j in jobs10])
        w["grid_wall_s"] = time.perf_counter() - t0
        w["grid_steps"] = int(max(len(s) for s, _ in batch))
        w["grid_rules_total"] = int(sum(len(s) for s, _ in batch))
        w["grid_max_equivalent"] = int(max((int(x["equiv_count"]) for s, _ in batch for x in s), default=0))
        t0 = time.perf_counter()
        alone = [b.scm_run([j[0]])[0] for j in jobs10]
        w["one_at_a_time_wall_s"] = time.perf_counter() - t0
        w["batched_equals_one_at_a_time"] = same(batch, alone)
        if G == 100:
            mat = b.matrix()
            ok = []
            for i in [104, 114, 100, 119][: args.oracle_fits]:          # full training set: conjunction / disjunction ...
                (job, pos, neg, p, mt), got = jobs10[i], batch[i]
                want = scm_fit(mat, G, pos.tolist(), neg.tolist(), ["conjunction", "disjunction"][mt], p, 10, (), True)
                steps, eq = got
                ok.append(len(steps) == len(want) and all(
                    int(s["rule"]) == x["rule"] and np.float64(s["utility"]).view(np.int64) == np.float64(x["utility"]).view(np.int64)
                    and int(s["positive_errors"]) == x["positive_errors"] and int(s["negative_covers"]) == x["negative_covers"]
                    and np.array_equal(eq[int(s["equiv_offset"]):int(s["equiv_offset"] + s["equiv_count"])].astype(np.int64), x["equivalent"])
                    for s, x in zip(steps, want)))
            w["oracle_fits_checked"] = len(ok)
            w["equals_oracle"] = all(ok)
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
