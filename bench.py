#!/usr/bin/env python
"""bench.py -- Gbases/s of the k-mer matrix build (k=31) on N B200s, with roofline, CPU baseline and parity check.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config auto|c1|c2|c3|c3w|c4|c5] [--dump-outputs DIR]
    python bench.py --impl reference [...]        CPU arm: the oracle port on the host cores (rank 0 only)
    (N > 1: launched by torch.distributed.run, one rank per GPU)

A "step" is one complete build of the workload: FASTA / FASTQ text -> packed stream -> minimizer-bounded units
(super-k-mers) -> content-hash buckets -> per-bucket dedupe across genomes -> k-mers of the distinct units -> hash
buckets -> shared-memory aggregation -> ordered columns (kmers[U] + matrix[W][U]); read sets with an abundance filter
run the front end in rounds of a few genomes with per-genome counters and end with one presence merge.
  value : whole-job Gbases/s with the text already resident in HBM (CUDA events, max over ranks)
  e2e   : same metric through the public API with HOST (pinned) buffers: H2D of the text and D2H of kmers + matrix
          inside the timed region, every step.  At N = 1 the steps run through builder.BuildPipeline (two contexts of the
          GPU alternate: step i+1's text goes in while step i's result comes out); e2e.serial is one build at a time
  parity_check : after the timed loops, the order-independent checksum of every rank's column slice (GPU kernel), summed
          over the ranks, against the same checksum of the oracle's matrix of the same genomes (rank 0, CPU)

Configs (BASELINE.json): c1 = 20 genomes, from-contigs (singletons dropped); c2 = 100 genomes, Ray Surveyor matrix
(singletons kept) -- the N = 1 default; c3 = 1,000 genomes over N GPUs (strong scaling); c3w = 125 genomes per GPU
(weak scaling: the N > 1 default, 1,000 genomes at N = 8); c4 = 200 read sets of 30x 150 bp reads, min abundance 2;
c5 = 500 genomes, k in {15, 21, 31} x singletons kept / dropped (one line with a sweep list).

--dump-outputs DIR: after the timed steps, a fixed, seeded sample of the columns of the last timed build goes to DIR as
.npy files (see dump_outputs), so that two builds of the project can be compared output for output: the inputs are the
same bytes on every run with the same arguments.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Gbases/s k-mer matrix build (k=31)"
UNIT = "Gbases/s"
K = 31
READS_PER_GENOME = 1_000_000      # 30x of a 5 Mbp genome at 150 bp
CPU_SAMPLE_BASES = 5.0e8          # bounded sample of the CPU arms: about 6 s on 16 cores
DUMP_BYTES = 48 << 20             # --dump-outputs: bytes of .npy data in all (the c5 sweep shares it among its builds)
DUMP_SEED = 1

CONFIGS = {
    "c1": dict(genomes=20, per_gpu=False, reads=False, min_ab=1, keep=False,
               label="C1: kover dataset create from-contigs, {g} synthetic 5 Mbp genomes, k=31, singletons dropped"),
    "c2": dict(genomes=100, per_gpu=False, reads=False, min_ab=1, keep=True,
               label="C2: Ray Surveyor genome x k-mer matrix, {g} synthetic 5 Mbp genomes, k=31, min abundance 1, singletons kept"),
    "c3": dict(genomes=1000, per_gpu=False, reads=False, min_ab=1, keep=True,
               label="C3: {g} synthetic 5 Mbp genomes k=31, rows sharded across {n} GPUs in 64-aligned blocks (strong scaling), "
                     "hash-range exchange (NVLink peer stores fused into the export kernel)"),
    "c3w": dict(genomes=125, per_gpu=True, reads=False, min_ab=1, keep=True,
                label="C3 family: {g} synthetic 5 Mbp genomes (125 per GPU) k=31, rows sharded across {n} GPUs in 64-aligned "
                      "blocks, hash-range exchange (NVLink peer stores fused into the export kernel)"),
    "c4": dict(genomes=200, per_gpu=False, reads=True, min_ab=2, keep=False,
               label="C4: from-reads, {g} synthetic read sets (30x, 150 bp, 0.5 % substitutions) k=31, min abundance 2, "
                     "singletons dropped, rows sharded across {n} GPUs"),
    "c5": dict(genomes=500, per_gpu=False, reads=False, min_ab=1, keep=False,
               label="C5: {g} synthetic 5 Mbp genomes, k sweep 15/21/31 x singletons kept/dropped (headline: k=31, dropped)"),
}


def pick_config(name, n_gpus):
    if name == "auto":
        name = "c2" if n_gpus == 1 else "c3w"
    return name, CONFIGS[name]


def total_genomes(conf, n_gpus, override):
    g = override or conf["genomes"]
    return g * n_gpus if conf["per_gpu"] else g


def workload_config(name, conf, n_gpus, G):
    return {"workload": conf["label"].format(g=G, n=n_gpus), "config": name, "genomes": G, "k": K,
            "min_abundance": conf["min_ab"], "keep_singletons": conf["keep"],
            "input": "FASTQ read sets, 1,000,000 reads x 150 bp per genome" if conf["reads"] else "FASTA contigs, 50 per genome",
            "l2": "inputs (>= 100 MB of text per GPU and step) larger than the 126 MB L2; no flush needed"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_from_profiles(kernel: str):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(p) as f:
            v = json.load(f).get(kernel)
            return v.get("dram_bytes_per_launch") if isinstance(v, dict) else v
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------------------------
# CPU side: the oracle port (restatement of multidsk + dsk2kover; the reference binaries are absent from the checkout,
# .MISSING_LARGE_BLOBS:1-4).  Checker-side code: only the cpu_baseline leg, --impl reference and parity_check run it.
# ---------------------------------------------------------------------------------------------------------------
def host_threads() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def cpu_arm(texts, kind, min_ab, keep, k=K):
    """One oracle build with every host thread.  -> (Gbases/s, seconds, threads, result)"""
    from oracle import oracle
    oracle.build_library()
    threads = host_threads()          # explicit: under torch.distributed.run OMP_NUM_THREADS defaults to 1
    t0 = time.perf_counter()
    r = oracle.build([[(t, kind)] for t in texts], k, min_ab, keep, threads=threads)
    dt = time.perf_counter() - t0
    return r.n_bases / dt / 1e9, dt, threads, r


def _synth_one(args):
    from grm_b200 import synth
    seed, g, reads = args
    cfg = synth.SynthConfig(seed=seed)
    return synth.genome_reads_fastq_fixed(cfg, g, READS_PER_GENOME) if reads else synth.genome_fasta(cfg, g)


def host_genomes(seed, ids, reads):
    """The workload's synthetic inputs made on the HOST (numpy mirror of the CUDA generator, identical bytes):
    the reference arm touches neither the GPU nor libgrmkm.so."""
    import multiprocessing as mp
    ids = list(ids)
    with mp.get_context("fork").Pool(min(host_threads(), max(1, len(ids)))) as pool:
        return pool.map(_synth_one, [(seed, g, reads) for g in ids])


def sample_ids(conf, G):
    per = 1.5e8 if conf["reads"] else 5.0e6
    return list(range(max(1, min(G, int(round(CPU_SAMPLE_BASES / per))))))


def run_reference(args):
    """--impl reference: the CPU implementation of the path on a bounded sample of the same workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from grm_b200 import synth
    n_gpus = int(os.environ.get("WORLD_SIZE", args.gpus))
    name, conf = pick_config(args.config, n_gpus)
    G = total_genomes(conf, n_gpus, args.genomes)
    ids = sample_ids(conf, G)
    texts = host_genomes(synth.MASTER_SEED + 1, ids, conf["reads"])
    kind = 1 if conf["reads"] else 0
    vals, times, threads = [], [], host_threads()
    budget_s, t_start = 240.0, time.perf_counter()
    for i in range(args.warmup + args.steps):
        v, dt, threads, ref = cpu_arm(texts, kind, conf["min_ab"], conf["keep"])
        if i >= args.warmup:
            vals.append(v); times.append(dt)
        if vals and time.perf_counter() - t_start > budget_s:
            break                                  # bounded: the arm must end within a few minutes whatever --steps says
    val = sum(vals) / len(vals)
    sample = (f"genomes 0..{len(ids) - 1} of the workload's {G} ({ref.n_bases} bases per step, "
              f"{'FASTQ read sets' if conf['reads'] else 'FASTA'}, k={K}, min abundance {conf['min_ab']}, singletons "
              f"{'kept' if conf['keep'] else 'dropped'}), {len(times)} timed steps of {args.steps} asked (240 s budget), "
              f"oracle port of multidsk+dsk2kover semantics with {threads} OpenMP threads; inputs made by the numpy generator")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": n_gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak" if conf["per_gpu"] else "strong", "vs_baseline": None, "dtype": "u64",
        "data": "synthetic", "config": workload_config(name, conf, n_gpus, G),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------------------
# GPU side
# ---------------------------------------------------------------------------------------------------------------
def device_genomes(builder, cfg, ids, reads=False):
    """Synthesise the genomes' FASTA / FASTQ on the device; returns (uint8 cuda tensor, spans, n_bases)."""
    import torch
    from grm_b200 import synth
    ids = list(ids)
    if reads:
        lay, total, spans = synth.build_reads_layout(cfg, ids, READS_PER_GENOME)
        n_bases = len(ids) * READS_PER_GENOME * 150
    else:
        lay, total, spans = synth.build_layout(cfg, ids)
        n_bases = synth.n_bases_of(cfg, ids)
    buf = torch.empty(max(total, 16), dtype=torch.uint8, device="cuda")
    if ids:
        builder._check(builder._lib.grmkm_synth_fasta_device(builder._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes,
                                                              C.c_void_p(buf.data_ptr()), total))
    return buf, spans, n_bases


def parity_check(db, cfg, conf, G_total, rank, world, dist, k, keep):
    """Order-independent checksum of (k-mer, column words): every rank's slice on its GPU, summed over the ranks, against
    the oracle's matrix of the same genomes (rank 0).  Read sets are too slow for the oracle at full size: a bounded
    subset is built separately on rank 0's GPU and compared (the ranks' checksums are still summed and reported)."""
    import numpy as np
    import torch
    from oracle import oracle
    cs = db.builder.checksum() if db.n_kmers else (0, 0)
    mine = torch.tensor([np.uint64(cs[0]).astype(np.int64), np.uint64(cs[1]).astype(np.int64), db.n_kmers],
                        dtype=torch.int64, device="cuda")
    if dist:
        allv = torch.empty(3 * world, dtype=torch.int64, device="cuda")
        torch.distributed.all_gather_into_tensor(allv, mine)
        allv = allv.view(world, 3).cpu().numpy()
    else:
        allv = mine.view(1, 3).cpu().numpy()
    if rank != 0:
        return None
    m64 = (1 << 64) - 1
    got = (sum(int(np.int64(v).astype(np.uint64)) for v in allv[:, 0]) & m64,
           sum(int(np.int64(v).astype(np.uint64)) for v in allv[:, 1]) & m64)
    U = int(allv[:, 2].sum())
    kind = 1 if conf["reads"] else 0
    t0 = time.perf_counter()
    out = {"checksum": ["%016x" % got[0], "%016x" % got[1]], "n_kmers": U}
    per_base_s = 1.0 / (0.075e9 * host_threads() / 16.0)
    full_bases = G_total * (1.5e8 if conf["reads"] else 5.0e6)
    if full_bases * per_base_s <= 400.0:
        texts = []
        for a in range(0, G_total, 64):
            buf, spans, _ = device_genomes(db.builder, cfg, range(a, min(G_total, a + 64)), conf["reads"])
            host = buf.cpu().numpy()
            texts.extend(host[o:o + n].tobytes() for o, n in spans)
            del buf, host
        ref = oracle.build([[(t, kind)] for t in texts], k, conf["min_ab"], keep, threads=host_threads())
        want = oracle.checksum(ref.kmers, ref.matrix)
        out.update({"ok": bool(want == got and ref.n_kmers == U), "against": "oracle (CPU restatement) over all genomes of the workload",
                    "genomes": G_total, "oracle_n_kmers": ref.n_kmers,
                    "oracle_checksum": ["%016x" % want[0], "%016x" % want[1]]})
    else:
        from grm_b200.builder import KmerMatrixBuilder
        n_sub = max(2, min(G_total, int(300.0 / (1.5e8 * per_base_s)) if conf["reads"] else 64))
        with KmerMatrixBuilder(k=k, min_abundance=conf["min_ab"], keep_singletons=keep, input_kind=kind) as b:
            buf, spans, _ = device_genomes(b, cfg, range(n_sub), conf["reads"])
            b.set_genome_count(n_sub)
            for row, (o, n) in enumerate(spans):
                b.add_genome_device(row, buf.data_ptr() + o, n)
            b.build()
            sub = b.checksum()
            sub_u = b.dims[0]
            host = buf.cpu().numpy()
        ref = oracle.build([[(host[o:o + n].tobytes(), kind)] for o, n in spans], k, conf["min_ab"], keep, threads=host_threads())
        want = oracle.checksum(ref.kmers, ref.matrix)
        out.update({"ok": bool(want == sub and ref.n_kmers == sub_u),
                    "against": f"oracle (CPU restatement) over genomes 0..{n_sub - 1}, built separately on rank 0's GPU "
                               "(the full workload is too slow for the CPU checker); the full result's checksum is reported",
                    "genomes": n_sub, "oracle_n_kmers": ref.n_kmers,
                    "oracle_checksum": ["%016x" % want[0], "%016x" % want[1]]})
    out["seconds"] = round(time.perf_counter() - t0, 1)
    return out


def e2e_files(texts, names, conf, k):
    """What a GRM user waits for: .fna files (tmpfs) -> from_contigs -> .kover file (gzip 4), wall clock."""
    import shutil
    import tempfile
    from grm_b200 import create, hdf5min
    d = tempfile.mkdtemp(prefix="grm_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        lines = []
        for n, t in zip(names, texts):
            p = os.path.join(d, n + ".fna")
            with open(p, "wb") as f:
                f.write(t)
            lines.append(f"{n}\t{p}\n")
        lst = os.path.join(d, "contigs.tsv")
        with open(lst, "w") as f:
            f.writelines(lines)
        out = os.path.join(d, "bench.kover")
        nbytes = sum(len(t) for t in texts)
        best = None
        for _ in range(2):
            t0 = time.perf_counter()
            create.from_contigs(lst, out, k, "nothing" if conf["keep"] else "singleton", None, None, 4, d, 0, False, False)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        U = hdf5min.H5Reader(out)["kmer_matrix"].shape[1]
        return {"seconds": best, "input_bytes": nbytes, "kover_bytes": os.path.getsize(out), "n_kmers": int(U), "gzip": 4,
                "what": ".fna files on tmpfs -> grm_b200.create.from_contigs -> .kover (HDF5, gzip 4, threaded zlib), best of 2"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


def dump_outputs(db, out_dir, prefix, n_genomes, budget, rank, world, dist):
    """Write a seeded sample of the columns of db's last build to out_dir/<prefix><name>.npy (rank 0; collective at N > 1):
      kmers   float32 [n][k]  bases of each sampled k-mer, first base first, in the 2-bit code of the packed k-mers
                              (A 0, C 1, T 2, G 3)
      matrix  float32 [G][n]  1 where genome g holds the k-mer, else 0
      columns float64 [n]     indices of the sampled columns in the result's column order (ascending)
      n_kmers float64 [1]     number of columns of the result
    Every value is a small integer, so a changed k-mer or presence bit differs by at least 1.  n is as many columns as
    `budget` bytes hold; the sample is drawn with DUMP_SEED from the column count alone."""
    import numpy as np
    counts = db.slice_counts()                   # the global column order is the ranks' slices in rank order
    U, off = sum(counts), sum(counts[:rank])
    n = min(U, budget // (4 * (db.k + n_genomes) + 8))
    cols = np.sort(np.random.default_rng(DUMP_SEED).choice(U, n, replace=False)) if n < U else np.arange(U)
    mine = cols[(cols >= off) & (cols < off + counts[rank])] - off
    km, mat = db.builder.kmers()[mine], db.builder.matrix()[:, mine]
    if world > 1:
        parts = [None] * world if rank == 0 else None
        dist.gather_object((km, mat), parts, dst=0)
        if rank != 0:
            return
        km, mat = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts], axis=1)
    shifts = np.uint64(2) * np.arange(db.k - 1, -1, -1, dtype=np.uint64)
    bases = (km[:, None] >> shifts) & np.uint64(3)
    # genome g is bit 63 - g % 64 of word row g // 64: the bits of the big-endian bytes, most significant first
    W = mat.shape[0]
    bits = np.unpackbits(np.ascontiguousarray(mat, dtype=">u8").view(np.uint8).reshape(W, n, 8), axis=2)
    presence = bits.transpose(0, 2, 1).reshape(W * 64, n)[:n_genomes]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("kmers", bases.astype(np.float32)), ("matrix", presence.astype(np.float32)),
                    ("columns", cols.astype(np.float64)), ("n_kmers", np.array([U], dtype=np.float64))):
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="grm_b200", choices=["grm_b200", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto"] + sorted(CONFIGS))
    ap.add_argument("--genomes", type=int, default=0, help="override the config's genome count (per GPU for c3w; debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-e2e-files", action="store_true")
    ap.add_argument("--no-e2e-pipeline", action="store_true", help="e2e with one context only (no builds in flight side by side)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a seeded sample of what the last timed build computed to DIR/*.npy (at most 48 MiB)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's result; the reference arm has none")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    from grm_b200 import synth
    from grm_b200.distributed import DistributedBuilder, init_process_group_from_env

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the k-mer matrix path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = init_process_group_from_env() if world > 1 else None
    if args.warmup < 3 and rank == 0:
        print("note: fewer than 3 warm-up steps; this run is for profiling, not a bench value", file=sys.stderr)

    name, conf = pick_config(args.config, world)
    G_total = total_genomes(conf, world, args.genomes)
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1)
    kind = 1 if conf["reads"] else 0
    stream = torch.cuda.Stream()
    peak, peak_src = peaks()
    sweep = [(K, conf["keep"])]
    if name == "c5":
        sweep = [(K, False), (K, True), (21, False), (21, True), (15, False), (15, True)]     # the headline first

    results = []
    with torch.cuda.stream(stream):
        buf = spans = None
        for si, (k, keep) in enumerate(sweep):
            db = DistributedBuilder(k=k, min_abundance=conf["min_ab"], keep_singletons=keep, n_genomes=G_total, rank=rank,
                                    world=world, input_kind=kind, stream=stream.cuda_stream, device=local_rank)
            my_rows = list(db.local_rows)                     # global genome rows of this rank
            if buf is None:
                buf, spans, my_bases = device_genomes(db.builder, cfg, my_rows, conf["reads"])
                stream.synchronize()
            rows_np = np.arange(len(spans), dtype=np.uint32)
            ptrs_np = np.array([buf.data_ptr() + off for off, _ in spans], dtype=np.uint64)
            lens_np = np.array([ln for _, ln in spans], dtype=np.uint64)

            def step_resident():
                db.reset()
                db.add_genomes(rows_np, ptrs_np, lens_np, on_device=True)
                db.build(reuse_partition=True)        # N > 1: the bucket count agreed in the first warm-up build is kept

            # ---- value: inputs resident in HBM
            for _ in range(args.warmup):
                step_resident()
            sampler = ClockSampler(local_rank)
            if rank == 0:
                sampler.start()
            if dist:
                torch.distributed.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            stage_acc, launches = {}, 0
            e0.record(stream)
            for _ in range(args.steps):
                step_resident()
                for kname, v in db.stage_times.items():
                    stage_acc[kname] = stage_acc.get(kname, 0.0) + v
                launches += db.launches
            e1.record(stream)
            torch.cuda.synchronize()
            if dist:
                torch.distributed.barrier()
            ms = e0.elapsed_time(e1)
            clocks = sampler.stop() if rank == 0 else None
            stats = dict(db.builder.stats)
            stats.update({k2: v for k2, v in db.local_stats.items() if k2 in (
                "n_windows", "n_input_bytes", "n_bases", "n_records", "n_buckets", "n_units", "n_unit_entries", "n_wide",
                "n_unit_buckets", "n_rounds", "n_solid_records")})
            if args.dump_outputs:
                dump_outputs(db, args.dump_outputs, "" if si == 0 else f"k{k}_{'kept' if keep else 'dropped'}_", G_total,
                             DUMP_BYTES // len(sweep), rank, world, dist)
            res = {"k": k, "keep": keep, "ms": ms, "stage_acc": stage_acc, "launches": launches, "stats": stats,
                   "U_local": db.n_kmers, "clocks": clocks, "ms_e2e": 0.0, "e2e_steps": 0, "h2d": 0, "d2h": 0, "parity": None}
            if si == 0:
                # ---- e2e: host (pinned) buffers in, kmers + matrix out, every step
                host_in, host_np = [], []
                res["h2d"] = sum(ln for _, ln in spans)

                def step_e2e():
                    db.reset()
                    db.add_genomes(rows_np, host_np)
                    db.build(reuse_partition=True)
                    return db.result_host()          # one D2H copy into the context's page-locked result buffer

                # page-locked staging on the GPU's own NUMA node (first touch under near_gpu, for the text here and for the
                # library's result buffer in the first step): no cross-socket hop per byte
                from grm_b200.numa import near_gpu
                with near_gpu(local_rank) as numa_node:
                    # one page-locked arena, files 16-byte aligned one after the other (what create._read_inputs makes of
                    # the .fna files): the library then moves a whole staging batch with one copy
                    offs, tot = [], 0
                    for _, ln in spans:
                        offs.append(tot)
                        tot += (ln + 15) & ~15
                    host_in = torch.zeros(max(tot, 16), dtype=torch.uint8).pin_memory()
                    for o, (off, ln) in zip(offs, spans):
                        host_in[o:o + ln].copy_(buf[off:off + ln])
                    stream.synchronize()
                    arena = host_in.numpy()
                    host_np = [arena[o:o + ln] for o, (_, ln) in zip(offs, spans)]
                    km, mat = step_e2e()
                res["numa_node"] = numa_node

                for _ in range(min(args.warmup, 2)):
                    km, mat = step_e2e()
                if dist:
                    torch.distributed.barrier()
                torch.cuda.synchronize()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                res["e2e_steps"] = max(1, min(args.steps, 5))
                f0.record(stream)
                for _ in range(res["e2e_steps"]):
                    km, mat = step_e2e()
                f1.record(stream)
                torch.cuda.synchronize()
                if dist:
                    torch.distributed.barrier()
                res["ms_e2e"] = f0.elapsed_time(f1)
                res["d2h"] = int(km.nbytes + mat.nbytes)
                res["ms_e2e_serial"], res["e2e_serial_steps"] = res["ms_e2e"], res["e2e_steps"]
                if world == 1 and not args.no_e2e_pipeline:
                    # a series of builds through the public BuildPipeline (two contexts of this GPU, one worker thread each):
                    # build i + 1's H2D copy runs while build i computes and copies its result out.  Every build copies its
                    # whole input in and its whole result out, as above.
                    from grm_b200.builder import BuildPipeline
                    ps = [torch.cuda.Stream() for _ in range(2)]
                    n_pipe = 2 * max(2, min(args.steps, 6) // 2 + 1)
                    with BuildPipeline(depth=2, streams=[s_.cuda_stream for s_ in ps], k=k, min_abundance=conf["min_ab"],
                                       keep_singletons=keep, input_kind=kind, device=local_rank) as pipe:
                        with near_gpu(local_rank):
                            for f_ in [pipe.submit(rows_np, host_np, n_genomes=G_total) for _ in range(4)]:
                                pk, pm, _ = f_.result()
                        if pk.shape != km.shape or not (np.array_equal(pk, km) and np.array_equal(pm, mat)):
                            raise SystemExit("bench.py: the pipelined build differs from the single-context build")
                        torch.cuda.synchronize()
                        g0 = torch.cuda.Event(enable_timing=True)
                        g0.record(ps[0])
                        for f_ in [pipe.submit(rows_np, host_np, n_genomes=G_total) for _ in range(n_pipe)]:
                            f_.result()
                        g1 = [torch.cuda.Event(enable_timing=True) for _ in ps]
                        for e_, s_ in zip(g1, ps):
                            e_.record(s_)
                        torch.cuda.synchronize()
                        res["ms_e2e"], res["e2e_steps"] = max(g0.elapsed_time(e_) for e_ in g1), n_pipe
                        res["e2e_mode"] = ("BuildPipeline(depth=2): two contexts of the GPU alternate, build i+1's H2D copy overlaps "
                                           "build i's tail kernels and D2H copy; every build copies its own input and result")
                if not args.no_parity_check:
                    res["parity"] = parity_check(db, cfg, conf, G_total, rank, world, dist, k, keep)
                if world == 1 and rank == 0 and not conf["reads"] and not args.no_e2e_files:
                    n_f = min(len(host_np), 100)
                    res["e2e_files"] = e2e_files([h.tobytes() for h in host_np[:n_f]], ["g%d" % g for g in my_rows[:n_f]], conf, k)
                    res["e2e_files"]["n_bases"] = synth.n_bases_of(cfg, my_rows[:n_f])
                del host_in, host_np
            results.append(res)
            if si + 1 < len(sweep):
                db.close()

    head = results[0]
    # ---- reduce over ranks: max time, sum bases
    tt = torch.tensor([head["ms"], head["ms_e2e"], float(my_bases), float(head["U_local"]), float(head["launches"]),
                       float(head["h2d"]), float(head["d2h"])] + [r["ms"] for r in results[1:]] + [float(r["U_local"]) for r in results[1:]],
                      dtype=torch.float64, device="cuda")
    if dist:
        mx = tt.clone(); torch.distributed.all_reduce(mx, op=torch.distributed.ReduceOp.MAX)
        sm = tt.clone(); torch.distributed.all_reduce(sm, op=torch.distributed.ReduceOp.SUM)
    else:
        mx = sm = tt
    ms, ms_e2e = float(mx[0]), float(mx[1])
    total_bases, U_total, launches = float(sm[2]), float(sm[3]), int(sm[4])
    h2d, d2h = int(sm[5]), int(sm[6])
    n_extra = len(results) - 1

    rc = 0
    if rank == 0:
        stats, stage_acc = head["stats"], head["stage_acc"]
        ms_step = ms / args.steps
        value = total_bases / (ms_step * 1e-3) / 1e9
        e2e_steps = head["e2e_steps"]
        e2e_val = total_bases / (ms_e2e / e2e_steps * 1e-3) / 1e9
        stage_ms = {k2: v / args.steps for k2, v in stage_acc.items()}
        # dominant kernel (rank 0's stage times; one launch per stage and round)
        W = stats["n_words"]
        n_in, U0 = stats["n_input_bytes"], stats["n_kmers"]
        stream_bytes = (stats["n_bases"] + stats["n_records"]) * 12 / 32
        # algorithmic bytes per launch (DESIGN.md section 4): the packed stream is 12 B and the run masks 8 B per 32
        # entries; a unit is 16 B; a dedupe entry (2 + WB) x 8 B; a wide record RS x 8 B
        n_units, n_ent, n_wide = stats.get("n_units", 0), stats.get("n_unit_entries", 0), stats.get("n_wide", 0)
        mask_bytes = (stats["n_bases"] + stats["n_records"]) * 8 / 32
        counting = conf["min_ab"] > 1
        WB = 1 if (W <= 1 or counting) else 2 if W == 2 else 4
        ent_b, rec_b = (2 + WB) * 8.0, (2 if WB == 1 else 2 * WB) * 8.0
        solid = stats.get("n_solid_records", 0)
        agg_out = 16.0 * solid + 16.0 * solid + U0 * 8.0 * (1 + W) if counting else U0 * 8.0 * (1 + W)
        kernels = {
            "k_units_scatter": (stage_ms.get("scatter", 0.0), stream_bytes + mask_bytes + 16.0 * n_units),
            "k_unit_bounds": (stage_ms.get("bounds", 0.0), stream_bytes + mask_bytes),
            "k_units_dedupe": (stage_ms.get("dedupe", 0.0), 16.0 * n_units + ent_b * n_ent),
            "k_units_expand": (stage_ms.get("expand", 0.0), 2 * ent_b * n_ent + rec_b * n_wide),
            "k_aggregate_cols": (stage_ms.get("aggregate", 0.0), rec_b * n_wide + agg_out),
            "k_pack": (stage_ms.get("pack", 0.0), n_in + stream_bytes),
        }
        dom = max(kernels, key=lambda n: kernels[n][0])
        dom_ms, dom_bytes = kernels[dom]
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        # whole-pipeline model of SURVEY.md 8d: B_alg = F + 8 + 8 + O bytes per base
        F = n_in / max(1, stats["n_bases"])
        O = U_total * (8 * ((G_total + 63) // 64) + 8) / total_bases
        b_alg = F + 16 + O
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak" if conf["per_gpu"] else "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": workload_config(name, conf, world, G_total),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": ms_e2e / e2e_steps, "staging_numa_node": head.get("numa_node"),
                    "mode": head.get("e2e_mode", "one build at a time (DistributedBuilder.build + result_host per step)"),
                    "serial": ({"value": total_bases / (head["ms_e2e_serial"] / head["e2e_serial_steps"] * 1e-3) / 1e9,
                                "ms_per_step": head["ms_e2e_serial"] / head["e2e_serial_steps"], "steps": head["e2e_serial_steps"],
                                "mode": "one build at a time"} if world == 1 and head.get("ms_e2e_serial") else None)},
            "gpu_launches": launches,
            "clocks": head["clocks"],
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic_from_profiles(dom), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": dom_bytes, "kernel_ms": dom_ms,
                         "kernel_share_of_step": dom_ms / ms_step if ms_step else None},
            "pipeline_roofline": {"bytes_per_base": b_alg, "achieved": value * b_alg, "peak": peak,
                                  "frac": value * b_alg / peak, "unit": "GB/s",
                                  "model": "SURVEY.md 8d: F + 8 + 8 + O bytes per base"},
            "stage_ms": stage_ms,
            "kernel_gbs": {n: (b / (t * 1e-3) / 1e9 if t > 0 else None) for n, (t, b) in kernels.items()},
            "result": {"n_bases": total_bases, "n_kmers": U_total, "n_genomes": G_total,
                       "n_buckets": stats["n_buckets"], "n_splits": stats["n_splits"],
                       "n_units": n_units, "n_unit_entries": n_ent, "n_wide_records": n_wide,
                       "n_unit_buckets": stats.get("n_unit_buckets", 0), "n_rounds": stats.get("n_rounds", 0),
                       "n_solid_records": solid},
            "parity_check": head["parity"],
        }
        if n_extra:
            line["sweep"] = [{"k": K, "keep_singletons": sweep[0][1], "value": value, "ms_per_step": ms_step, "n_kmers": U_total}]
            for i, r in enumerate(results[1:]):
                ms_i = float(mx[7 + i]) / args.steps
                line["sweep"].append({"k": r["k"], "keep_singletons": r["keep"], "value": total_bases / (ms_i * 1e-3) / 1e9,
                                      "ms_per_step": ms_i, "n_kmers": float(sm[7 + n_extra + i])})
        if "e2e_files" in head:
            ef = head["e2e_files"]
            ef["value"] = ef["n_bases"] / ef["seconds"] / 1e9
            ef["unit"] = UNIT
            line["e2e_files"] = ef
        if world == 1 and not args.no_cpu_baseline:
            ids = sample_ids(conf, len(spans))
            host = buf[:spans[ids[-1]][0] + spans[ids[-1]][1]].cpu().numpy()
            texts = [host[o:o + n].tobytes() for o, n in (spans[i] for i in ids)]
            v, dt, threads, ref = cpu_arm(texts, kind, conf["min_ab"], conf["keep"])
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"first {len(ids)} genomes of the workload ({ref.n_bases} bases), "
                                              f"oracle port of multidsk+dsk2kover semantics, {dt:.1f} s"}
        print(json.dumps(line))
        if head["parity"] is not None and not head["parity"].get("ok"):
            print("parity_check FAILED: the GPU result's checksum differs from the oracle's", file=sys.stderr)
            rc = 3
    db.close()
    if dist:
        code = torch.tensor([rc], device="cuda")
        torch.distributed.broadcast(code, src=0)
        rc = int(code.item())
        torch.distributed.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
