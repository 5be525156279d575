"""N ranks under a real torchrun launch, CUDA kernels on every rank (-m gpu).

With >= 2 GPUs the ranks use NCCL and the NVLink peer export; on a one-GPU box the two ranks share the device and
the transport is gloo (the partial columns cross the host), everything else -- partial builds, owner ranges, the
owner-side merge kernels, slice files / TSV offsets -- is the same code.  The results must be the bytes of a one-GPU
build."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle
from tests import inputs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _write_genomes(tmp_path, rng, G, reads=False):
    shared = [inputs.rand_seq(rng, 6000), inputs.rand_seq(rng, 1500)]
    paths = []
    for g in range(G):
        if reads:
            d = tmp_path / f"reads_{g}"
            d.mkdir()
            (d / "a.fastq").write_bytes(inputs.fastq(rng, shared[g % 2], n_reads=500, read_len=80))
            paths.append(str(d))
        else:
            p = tmp_path / f"genome_{g}.fna"
            p.write_bytes(inputs.fasta(rng, n_records=3, max_len=900, shared=shared))
            paths.append(str(p))
    return paths


def _datasets(path):
    from grm_b200 import hdf5min
    r = hdf5min.H5Reader(str(path))
    return {n: r[n].read() for n in ("kmer_matrix", "kmer_sequences", "genome_identifiers", "kmer_by_matrix_column")}, r.attrs


@pytest.mark.parametrize("ranks", [2, 3])
def test_from_contigs_on_n_ranks_writes_the_one_gpu_file(gpu, tmp_path, ranks):
    from grm_b200 import create
    rng = np.random.default_rng(ranks)
    G = 150                                               # three matrix word rows: 2 + 1 (two ranks), 1 + 1 + 1 (three)
    paths = _write_genomes(tmp_path, rng, G)
    lst = tmp_path / "contigs.tsv"
    lst.write_text("".join(f"g{g}\t{p}\n" for g, p in enumerate(paths)))
    md = tmp_path / "md.tsv"
    md.write_text("".join(f"g{g}\t{'RS'[g % 2]}\n" for g in range(G)))
    kw = dict(kmer_size=21, filter_singleton="singleton", phenotype_description="pheno", phenotype_metadata_path=str(md),
              gzip=1, temp_dir=str(tmp_path), nb_cores=2, verbose=False, progress=False)
    create.from_contigs(str(lst), str(tmp_path / "one.kover"), **kw)
    create.from_contigs(str(lst), str(tmp_path / "multi.kover"), gpus=ranks, **kw)
    a, attrs_a = _datasets(tmp_path / "one.kover")
    b, attrs_b = _datasets(tmp_path / "multi.kover")
    for name in a:
        assert a[name].dtype == b[name].dtype and np.array_equal(a[name], b[name]), name
    for key in attrs_a:                                   # everything but the time stamp and the uuid
        if key not in ("created", "uuid"):
            assert attrs_a[key] == attrs_b[key], key


def test_from_reads_with_abundance_filter_on_two_ranks(gpu, tmp_path, monkeypatch):
    from grm_b200 import create
    rng = np.random.default_rng(9)
    G = 70
    dirs = _write_genomes(tmp_path, rng, G, reads=True)
    lst = tmp_path / "reads.tsv"
    lst.write_text("".join(f"g{g}\t{p}\n" for g, p in enumerate(dirs)))
    kw = dict(kmer_size=25, abundance_min=2, filter_singleton="nothing", phenotype_description=None,
              phenotype_metadata_path=None, gzip=0, temp_dir=str(tmp_path), nb_cores=2, verbose=False, progress=False)
    create.from_reads(str(lst), str(tmp_path / "one.kover"), **kw)
    monkeypatch.setenv("GRM_GPUS", "2")                   # the environment switch instead of the keyword
    create.from_reads(str(lst), str(tmp_path / "multi.kover"), **kw)
    a, _ = _datasets(tmp_path / "one.kover")
    b, _ = _datasets(tmp_path / "multi.kover")
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    files = [[(open(os.path.join(d, "a.fastq"), "rb").read(), 1)] for d in dirs]
    ref = oracle.build(files, 25, 2, True)
    assert np.array_equal(b["kmer_matrix"], ref.matrix)


def test_surveyor_tsv_written_by_two_ranks(gpu, tmp_path):
    from grm_b200 import surveyor
    rng = np.random.default_rng(17)
    G = 90
    paths = _write_genomes(tmp_path, rng, G)
    out1, out2 = tmp_path / "o1", tmp_path / "o2"
    out1.mkdir(); out2.mkdir()
    c1 = surveyor.generate_survey_conf(paths, 31, str(out1))
    c2 = surveyor.generate_survey_conf(paths, 31, str(out2))
    p1 = surveyor.run_surveyor(c1)
    p2 = surveyor.run_surveyor(c2, gpus=2)
    a, b = open(p1, "rb").read(), open(p2, "rb").read()
    assert a == b
    ref = oracle.build([[(open(p, "rb").read(), 0)] for p in paths], 31, 1, True,
                       want_tsv_names=[os.path.splitext(os.path.basename(p))[0] for p in paths])
    assert b == ref.tsv


def test_bench_parity_check_under_torchrun(gpu, tmp_path):
    """bench.py at N = 2 under torch.distributed.run: the line must carry parity_check.ok (GPU checksum of the ranks'
    slices, summed, against the oracle's matrix of the same genomes), and --dump-outputs must hold the oracle's k-mers
    and presence bits at the sampled columns.  Needs two GPUs (NCCL refuses two ranks on one device); on a one-GPU box
    the N = 1 line is checked instead."""
    import torch
    from grm_b200 import synth
    n = 2 if torch.cuda.device_count() >= 2 else 1
    cmd = [sys.executable]
    if n > 1:
        cmd += ["-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
                "--master-port", "29533"]
    out = tmp_path / "outputs"
    cmd += [os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--steps", "2", "--warmup", "1", "--genomes", "6",
            "--no-cpu-baseline", "--dump-outputs", str(out)]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["n_gpus"] == n and line["parity_check"]["ok"] is True, line.get("parity_check")
    assert line["parity_check"]["against"].startswith("oracle")

    c = line["config"]
    G, k = c["genomes"], c["k"]
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1)           # bench.py's inputs, made on the host
    ref = oracle.build([[(synth.genome_fasta(cfg, g), 0)] for g in range(G)], k, c["min_abundance"], c["keep_singletons"])
    d = {name: np.load(out / f"{name}.npy") for name in ("kmers", "matrix", "columns", "n_kmers")}
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    assert d["kmers"].dtype == d["matrix"].dtype == np.float32 and d["columns"].dtype == np.float64
    assert d["n_kmers"].tolist() == [ref.n_kmers]
    cols = d["columns"].astype(np.int64)
    assert 0 < len(cols) and np.all(np.diff(cols) > 0) and cols[-1] < ref.n_kmers
    assert d["kmers"].shape == (len(cols), k) and d["matrix"].shape == (G, len(cols))
    packed = np.zeros(len(cols), dtype=np.uint64)
    for i in range(k):
        packed = (packed << np.uint64(2)) | d["kmers"][:, i].astype(np.uint64)
    assert np.array_equal(packed, ref.kmers[cols])
    g = np.arange(G)
    bits = (ref.matrix[g // 64][:, cols] >> (np.uint64(63) - (g % 64).astype(np.uint64))[:, None]) & np.uint64(1)
    assert np.array_equal(d["matrix"], bits.astype(np.float32))
