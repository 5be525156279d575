"""grmkm_query: the genomes' rows against a k-mer set without a build.  Times the query on device-resident text, the
composition available without it (a build with singletons kept, then a host lookup of the same k-mers in its
columns), and one query end to end from page-locked host memory; checks bit for bit that the query columns equal the
build's.  Prints one JSON line (commit it under profiles/).

Workloads: synthetic 5 Mbp genomes of synth.py generated on the GPU, as tools/scm_bench.py -- C2's shape (100 genomes)
and 500 genomes, k = 31.  Query sizes Q = 10 / 1 000 / 100 000 / 1 000 000: half drawn from the build's columns, half
at random.  Times are medians over at least --min-seconds of repeated calls (device time from the call's CUDA events,
and wall time of the call, which ends in a synchronize).

    python tools/query_bench.py [--out FILE] [--min-seconds 0.5]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from scm_bench import card  # noqa: E402

WORKLOADS = [("c2_100_genomes", 100), ("500_genomes", 500)]
Q_SIZES = [10, 1_000, 100_000, 1_000_000]


def synth_text(G):
    import torch
    from grm_b200 import synth
    from grm_b200.builder import KmerMatrixBuilder
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1)
    lay, total, spans = synth.build_layout(cfg, list(range(G)))
    buf = torch.empty(max(total, 16), dtype=torch.uint8, device="cuda")
    with KmerMatrixBuilder(k=31) as b:
        b._check(b._lib.grmkm_synth_fasta_device(b._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes,
                                                 C.c_void_p(buf.data_ptr()), total))
    torch.cuda.synchronize()
    return buf, spans


def device_builder(buf, spans, G, **kw):
    from grm_b200.builder import KmerMatrixBuilder
    b = KmerMatrixBuilder(k=31, **kw)
    b.set_genome_count(G)
    b.add_genomes(np.arange(G, dtype=np.uint32), np.array([buf.data_ptr() + o for o, _ in spans], dtype=np.uint64),
                  np.array([n for _, n in spans], dtype=np.uint64), on_device=True)
    return b


def repeat(fn, min_s):
    fn()                                                  # warm-up: modules, buffers, the shape of this call
    walls, devs = [], []
    t_end = time.perf_counter() + min_s
    while time.perf_counter() < t_end or len(walls) < 3:
        t0 = time.perf_counter()
        dev = fn()
        walls.append((time.perf_counter() - t0) * 1e3)
        devs.append(dev)
    return float(np.median(walls)), (float(np.median(devs)) if devs[0] is not None else None), len(walls)


def canonical(x):
    x = np.asarray(x, dtype=np.uint64)
    rc = np.zeros_like(x)
    f = x.copy()
    for _ in range(31):
        rc = (rc << np.uint64(2)) | ((f & np.uint64(3)) ^ np.uint64(2))
        f >>= np.uint64(2)
    return np.minimum(x, rc)


def lookup(kmers, mat, q):
    """the composition's host step: the columns of q's canonical k-mers in a keep-singletons build, zeros elsewhere"""
    order = np.argsort(kmers)
    sk = kmers[order]
    c = canonical(q)
    pos = np.minimum(np.searchsorted(sk, c), len(sk) - 1)
    found = sk[pos] == c
    out = np.zeros((mat.shape[0], len(q)), dtype=np.uint64)
    out[:, found] = mat[:, order[pos[found]]]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--min-seconds", type=float, default=0.5)
    args = ap.parse_args()
    import torch
    res = {"tool": "query_bench", "card": card(), "k": 31, "min_seconds": args.min_seconds, "workloads": {}}
    ok = True
    rng = np.random.default_rng(5)
    for name, G in WORKLOADS:
        buf, spans = synth_text(G)
        text = int(sum(n for _, n in spans))
        w = {"genomes": G, "text_bytes": text, "queries": {}}
        with device_builder(buf, spans, G, keep_singletons=True) as b:
            b.build()
            kmers, mat = b.kmers(), b.matrix()
            bs = b.stats
            w.update(columns=int(len(kmers)), n_bases=int(bs["n_bases"]), n_windows=int(bs["n_windows"]))

            def compose(q):
                t0 = time.perf_counter()
                b.build()
                out = lookup(b.kmers(), b.matrix(), q)
                return out, (time.perf_counter() - t0) * 1e3

            lo = min(o for o, _ in spans)
            hi = max(o + n for o, n in spans)
            pinned = torch.empty(max(hi - lo, 16), dtype=torch.uint8, pin_memory=True)
            pinned[:hi - lo].copy_(buf[lo:hi])
            host = pinned.numpy()
            for Q in Q_SIZES:
                half = Q // 2
                q = np.concatenate([kmers[rng.choice(len(kmers), size=half, replace=False)],
                                    rng.integers(0, 2**62, size=Q - half, dtype=np.uint64)]).astype(np.uint64)
                got, st = b.query(q, with_stats=True)
                want, _ = compose(q)
                exact = bool(np.array_equal(got, want))
                ok &= exact
                wall, dev, reps = repeat(lambda: b.query(q, with_stats=True)[1]["ms"], args.min_seconds)
                c_wall, _, c_reps = repeat(lambda: (compose(q), None)[1], args.min_seconds)
                from grm_b200.builder import KmerMatrixBuilder
                with KmerMatrixBuilder(k=31) as hb:
                    hb.set_genome_count(G)
                    hb.add_genomes(np.arange(G, dtype=np.uint32), [host[o - lo:o - lo + n] for o, n in spans])
                    h_exact = bool(np.array_equal(hb.query(q), got))
                    ok &= h_exact
                    h_wall, h_dev, h_reps = repeat(lambda: hb.query(q, with_stats=True)[1]["ms"], args.min_seconds)
                groups = (int(bs["n_bases"]) + int(bs["n_records"])) / 32
                w["queries"][str(Q)] = {
                    "n_queries": st["n_queries"], "n_hits": st["n_hits"], "n_jobs": st["n_jobs"],
                    "tier": "shared" if st["n_queries"] <= 4096 else "global",
                    "query_device_ms": dev, "query_wall_ms": wall, "query_reps": reps,
                    "query_gbases_per_s": st["n_bases"] / (dev * 1e-3) / 1e9,
                    "compose_build_lookup_wall_ms": c_wall, "compose_reps": c_reps,
                    "host_query_device_ms": h_dev, "host_query_wall_ms": h_wall, "host_query_reps": h_reps,
                    "host_query_gbases_per_s": st["n_bases"] / (h_dev * 1e-3) / 1e9,
                    "bit_exact_vs_build": exact, "host_equals_device": h_exact,
                }
            # HBM bytes per base of a device-resident query: the pack reads the text and writes the packed stream
            # (8 B codes + 4 B validity per 32 entries), the scan reads the stream
            w["hbm_bytes_per_base"] = (text + 2 * 12 * groups) / int(bs["n_bases"])
            del pinned, host
        del buf
        torch.cuda.empty_cache()
        res["workloads"][name] = w
    res["ok"] = bool(ok)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
