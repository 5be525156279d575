"""grmkm_query on the GPU (-m gpu): the genomes' rows against a k-mer set without a build, bit for bit against the
oracle's per-genome solid sets and against the matrix of a build; read sets, both table tiers, forced batch and row
splits, no side effects on the context, the refusals, and predict_genomes against predict."""
import ctypes as C
import gzip
import os

import numpy as np
import pytest

from oracle import oracle
from tests import inputs
from tests.test_gpu_scm import _insert_genomes

pytestmark = pytest.mark.gpu

SMEM_KEYS = 4096          # kQuerySmemKeys (grmkm_query.cuh): the largest set whose table sits in shared memory


def canon(x, k):
    """canonical k-mers of a packed array (or one value)"""
    x = np.asarray(x, dtype=np.uint64)
    rc, f = np.zeros_like(x), x.copy()
    for _ in range(k):
        rc = (rc << np.uint64(2)) | ((f & np.uint64(3)) ^ np.uint64(2))
        f >>= np.uint64(2)
    return np.minimum(x, rc)


def revcomp(x, k):
    x = int(x)
    rc = 0
    for _ in range(k):
        rc = (rc << 2) | ((x & 3) ^ 2)
        x >>= 2
    return rc


def expected(files, G, kmers, k, min_ab=1):
    """files: row -> list of (bytes, kind).  The plane of the oracle's per-genome solid sets, and n_bases / n_windows."""
    can = canon(kmers, k)
    out = np.zeros(((G + 63) // 64, len(kmers)), dtype=np.uint64)
    nb = nw = 0
    for g in range(G):
        if not files.get(g):
            continue
        km, _, b, w = oracle.genome_solid(files[g], k, min_ab)
        nb += b
        nw += w
        hit = np.isin(can, km)
        out[g // 64, hit] |= np.uint64(1) << np.uint64(63 - g % 64)
    return out, nb, nw


def make_builder(files, G, k, min_ab=1, kind=0, keep=False):
    from grm_b200.builder import KmerMatrixBuilder
    b = KmerMatrixBuilder(k=k, min_abundance=min_ab, keep_singletons=keep, input_kind=kind)
    b.set_genome_count(G)
    for g, fs in files.items():
        for data, _ in fs:
            b.add_genome_bytes(g, data)
    return b


def query_set(rng, files, k, G, n_absent=50):
    """present k-mers on both strands, absent ones, duplicates"""
    present = []
    for g in sorted(files)[:20]:
        km, _, _, _ = oracle.genome_solid(files[g], k, 1)
        if len(km):
            present += [int(x) for x in rng.choice(km, size=min(10, len(km)), replace=False)]
    present = [revcomp(x, k) if i % 2 else x for i, x in enumerate(present)]
    lim = 1 << (2 * k)
    absent = [int(x) % lim for x in rng.integers(0, 2**63, size=n_absent)]
    q = present + absent + present[:5] + absent[:3]
    rng.shuffle(q)
    return np.array(q, dtype=np.uint64)


def fasta_genomes(rng, G, n_files=lambda g: 1, empty_every=0):
    files = {}
    for g in range(G):
        if empty_every and g % empty_every == empty_every - 1:
            continue                                            # a row without input
        fs = []
        for f in range(n_files(g)):
            if (g + f) % 11 == 5:
                fs.append((b"", 0))                            # an empty file
                continue
            fs.append((inputs.fasta(rng, n_records=int(rng.integers(1, 4)), max_len=300, crlf=bool(g % 3 == 1),
                                    blank=bool(g % 4 == 2), final_nl=bool(g % 5 != 3)), 0))
        files[g] = fs
    return files


@pytest.mark.parametrize("k", [1, 5, 11, 21, 31, 32])
@pytest.mark.parametrize("G", [1, 63, 64, 65, 300])
def test_against_the_oracle_genome_by_genome(gpu, G, k):
    rng = np.random.default_rng(G * 100 + k)
    files = fasta_genomes(rng, G, n_files=lambda g: 1 + (g % 3 == 0), empty_every=7 if G > 1 else 0)
    G_decl = G + (3 if G > 1 else 0)                           # trailing rows from set_genome_count
    q = query_set(rng, files, k, G)
    want, nb, nw = expected(files, G_decl, q, k)
    with make_builder(files, G_decl, k) as b:
        got, st = b.query(q, with_stats=True)
        assert got.shape == ((G_decl + 63) // 64, len(q))
        assert np.array_equal(got, want)
        assert (st["n_bases"], st["n_windows"]) == (nb, nw)
        assert st["n_queries"] == len(np.unique(canon(q, k)))
        assert st["n_input_bytes"] == sum(len(d) for fs in files.values() for d, _ in fs)
        assert st["n_jobs"] == 1 and st["ms"] > 0
        assert b.query(q[:0]).shape == ((G_decl + 63) // 64, 0)
        assert np.array_equal(b.query(q[:1]), want[:, :1])


def read_sets(rng, G):
    src = [inputs.rand_seq(rng, 600) for _ in range(3)]
    return {g: [(inputs.fastq(rng, src[g % 3], n_reads=150, read_len=40, crlf=bool(g % 2)), 1)] for g in range(G)}


@pytest.mark.parametrize("min_ab", [1, 2, 3])
def test_read_sets(gpu, tmp_path, min_ab):
    from grm_b200.builder import FASTQ, KmerMatrixBuilder
    rng = np.random.default_rng(40 + min_ab)
    G, k = 70, 21
    files = read_sets(rng, G)
    q = query_set(rng, files, k, G)
    want, nb, nw = expected(files, G, q, k, min_ab)
    with make_builder(files, G, k, min_ab, kind=FASTQ) as b:
        got, st = b.query(q, with_stats=True)
        assert np.array_equal(got, want)
        assert (st["n_bases"], st["n_windows"]) == (nb, nw)
    # the same reads from .gz files
    with KmerMatrixBuilder(k=k, min_abundance=min_ab, input_kind=FASTQ) as b:
        for g, fs in files.items():
            p = tmp_path / f"r{g}.fastq.gz"
            p.write_bytes(gzip.compress(fs[0][0]))
            b.add_genome_files(g, [str(p)])
        assert np.array_equal(b.query(q), want)


def present_and_absent(rng, files, k, n):
    pool = np.unique(np.concatenate([oracle.genome_solid(fs, k, 1)[0] for fs in files.values()]))
    take = rng.choice(pool, size=min(n // 2, len(pool)), replace=False)
    rand = np.unique(canon(rng.integers(0, 2**62, size=2 * n, dtype=np.uint64), k))
    rand = rng.permutation(rand[~np.isin(rand, pool)])[:n - len(take)]
    return np.concatenate([take, rand]).astype(np.uint64)


@pytest.mark.parametrize("Q", [SMEM_KEYS, SMEM_KEYS + 1, 1_000_000])
def test_both_table_tiers(gpu, Q):
    rng = np.random.default_rng(Q)
    G, k = 65, 31
    files = fasta_genomes(rng, G)
    q = present_and_absent(rng, files, k, Q)
    assert len(np.unique(canon(q, k))) == Q
    want, _, _ = expected(files, G, q, k)
    with make_builder(files, G, k) as b:
        got, st = b.query(q, with_stats=True)
        assert st["n_queries"] == Q
        assert np.array_equal(got, want)
        os.environ["GRMKM_QUERY_GLOBAL"] = "1"                # the global-memory table for a small set too
        try:
            assert np.array_equal(b.query(q), want)
        finally:
            del os.environ["GRMKM_QUERY_GLOBAL"]


@pytest.mark.parametrize("min_ab,kind", [(1, 0), (2, 1)])
def test_forced_batch_and_row_splits(gpu, min_ab, kind):
    rng = np.random.default_rng(50 + min_ab)
    G, k = 200, 21
    files = fasta_genomes(rng, G, empty_every=9) if kind == 0 else read_sets(rng, G)
    q = query_set(rng, files, k, G)
    with make_builder(files, G, k, min_ab, kind=kind) as b:
        one = b.query(q)
        assert one.any() and np.array_equal(one, expected(files, G, q, k, min_ab)[0])
        for rows in ("1", "64", "65"):
            os.environ["GRMKM_QUERY_ROWS"] = rows
            try:
                got, st = b.query(q, with_stats=True)
            finally:
                del os.environ["GRMKM_QUERY_ROWS"]
            assert np.array_equal(got, one), rows
            assert st["n_jobs"] > 1
    os.environ["GRMKM_BATCH_BYTES"] = "3000"                   # many pipelined batches (read at context creation)
    try:
        with make_builder(files, G, k, min_ab, kind=kind) as b:
            assert np.array_equal(b.query(q), one)
    finally:
        del os.environ["GRMKM_BATCH_BYTES"]


def test_against_a_build_at_the_c2_shape(gpu):
    import torch
    from grm_b200 import synth
    from grm_b200.builder import KmerMatrixBuilder
    G = 100
    cfg = synth.SynthConfig(seed=synth.MASTER_SEED + 1)
    lay, total, spans = synth.build_layout(cfg, list(range(G)))
    with KmerMatrixBuilder(k=31, keep_singletons=True) as b:
        buf = torch.empty(max(total, 16), dtype=torch.uint8, device="cuda")
        b._check(b._lib.grmkm_synth_fasta_device(b._ctx, C.c_void_p(lay.ctypes.data), lay.nbytes,
                                                 C.c_void_p(buf.data_ptr()), total))
        torch.cuda.synchronize()
        b.set_genome_count(G)
        b.add_genomes(np.arange(G, dtype=np.uint32), np.array([buf.data_ptr() + o for o, _ in spans], dtype=np.uint64),
                      np.array([n for _, n in spans], dtype=np.uint64), on_device=True)
        b.build()
        kmers, mat = b.kmers(), b.matrix()
        n = min(1_000_000, len(kmers))
        got, st = b.query(kmers[:n], with_stats=True)
        assert np.array_equal(got, mat[:, :n])
        assert st["n_windows"] == b.stats["n_windows"] and st["n_bases"] == b.stats["n_bases"]
        del buf


def _fitted(rc, pos, neg):
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.cart import fit_many as cart_many
    from grm_b200.scm import SetCoveringMachine
    from grm_b200.scm import fit_many as scm_many
    ms = [SetCoveringMachine(t, p, 4) for t in ("conjunction", "disjunction") for p in (0.5, 1.0, 5.0)]
    scm_many(rc, [(m, pos, neg) for m in ms])
    ts = [DecisionTreeClassifier(max_depth=d, class_importance=ci)
          for d, ci in ((3, None), (None, {0: 1.0, 1: 2.5}), (2, {0: 0.3, 1: 1.0}))]
    cart_many(rc, [(t, pos, neg) for t in ts])
    return ms + ts


def test_no_side_effects(gpu):
    from grm_b200 import native
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(60)
    insert = inputs.rand_seq(rng, 100)
    G, k = 80, 21
    genomes, carriers = _insert_genomes(rng, G, insert)
    files = {g: [(fa, 0)] for g, fa in enumerate(genomes)}
    with make_builder(files, G, k) as b:
        b.build()
        rc = KmerRuleClassifications(b, G)
        pos, neg = np.nonzero(carriers)[0], np.nonzero(~carriers)[0]
        models = _fitted(rc, pos, neg)
        assert len(models) == 9

        def fits():
            got = []
            for fn, cls, n in (("grmkm_scm_result", native.ScmStep, 6), ("grmkm_cart_result", native.CartNode, 3)):
                for f in range(n):
                    ns, ne = C.c_uint64(), C.c_uint64()
                    getattr(b._lib, fn)(b._ctx, f, None, 0, C.byref(ns), None, 0, C.byref(ne))
                    steps, eq = (cls * max(1, ns.value))(), np.zeros(max(1, ne.value), dtype=np.uint64)
                    assert getattr(b._lib, fn)(b._ctx, f, C.byref(steps), ns.value, C.byref(ns), C.c_void_p(eq.ctypes.data),
                                               ne.value, C.byref(ne)) == native.OK
                    got.append((bytes(steps), eq.tobytes()))
            return got

        # (stats right around the query: the checksum's own kernel counts in n_launches)
        q = query_set(rng, files, k, G)
        kept = (b.kmers(), b.matrix(), b.checksum(), fits())
        before = (b.stats, b.times) + kept
        b.query(q)
        after = (b.stats, b.times, b.kmers(), b.matrix(), b.checksum(), fits())
        assert np.array_equal(before[2], after[2]) and np.array_equal(before[3], after[3])
        assert before[1] == after[1] and before[4:] == after[4:]
        # (device_bytes is the memory the context holds now, which counts the buffers the query keeps for the next one)
        assert {**before[0], "device_bytes": 0} == {**after[0], "device_bytes": 0}
        # a build after a query gives the bytes of a build in a fresh context
        b.query(q)
        b.build()
        km2, mat2 = b.kmers(), b.matrix()
    with make_builder(files, G, k) as fresh:
        fresh.build()
        assert np.array_equal(fresh.kmers(), km2) and np.array_equal(fresh.matrix(), mat2)


def test_refusals(gpu):
    from grm_b200 import native
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(70)
    G, k = 10, 11
    files = fasta_genomes(rng, G)
    q = query_set(rng, files, k, G)
    want, _, _ = expected(files, G, q, k)
    with make_builder(files, G, k) as b:
        lib, ctx = b._lib, b._ctx
        out = np.zeros((1, len(q)), dtype=np.uint64)
        bad = q.copy()
        bad[3] = 1 << (2 * k)
        assert lib.grmkm_query(ctx, C.c_void_p(bad.ctypes.data), len(bad), C.c_void_p(out.ctypes.data), out.size, None) \
            == native.E_INVALID
        st = native.QueryStats()
        st.struct_size = 12
        assert lib.grmkm_query(ctx, C.c_void_p(q.ctypes.data), len(q), C.c_void_p(out.ctypes.data), out.size,
                               C.byref(st)) == native.E_INVALID
        assert lib.grmkm_query(ctx, C.c_void_p(q.ctypes.data), len(q), C.c_void_p(out.ctypes.data), out.size - 1,
                               None) == native.E_CAPACITY
        assert lib.grmkm_query(ctx, C.c_void_p(q.ctypes.data), len(q), C.c_void_p(out.ctypes.data), out.size,
                               None) == native.OK
        assert np.array_equal(out, want)
        assert np.array_equal(b.query(q), want)
    with KmerMatrixBuilder(k=k, flags=native.FLAG_COUNTS) as b:
        b.add_genome_bytes(0, files[0][0][0])
        with pytest.raises(native.GrmkmError) as e:
            b.query(q)
        assert e.value.code == native.E_INVALID
    with KmerMatrixBuilder(k=k) as b:                         # G = 0
        assert b.query(q).shape == (0, len(q))


def _end_to_end(rc, train_pos, train_neg, rows_b, b2):
    from grm_b200.predict import predict_genomes
    models = _fitted(rc, train_pos, train_neg)
    assert any(len(m.model) for m in models[:6]) and any(len(m.nodes) > 1 for m in models[6:])
    together = predict_genomes(models, b2)
    for m, got in zip(models, together):
        want = m.predict(rc, rows_b)
        assert np.array_equal(got, want)
        assert np.array_equal(m.predict_genomes(b2), want)


@pytest.mark.parametrize("kind", ["fasta", "fastq"])
def test_predict_genomes_equals_predict(gpu, kind):
    from grm_b200.builder import FASTQ, KmerMatrixBuilder
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(80)
    insert = inputs.rand_seq(rng, 150)
    G, k = 90, 21
    genomes, carriers = _insert_genomes(rng, G, insert)
    min_ab, ik = 1, 0
    if kind == "fastq":
        genomes = [inputs.fastq(rng, fa.split(b"\n", 1)[1].replace(b"\n", b""), n_reads=400, read_len=60, err=0.002)
                   for fa in genomes]
        min_ab, ik = 2, FASTQ
    a_rows, b_rows = np.arange(0, 60), np.arange(60, G)
    labels = carriers ^ (rng.random(G) < 0.1)
    with KmerMatrixBuilder(k=k, min_abundance=min_ab, input_kind=ik) as b, \
            KmerMatrixBuilder(k=k, min_abundance=min_ab, input_kind=ik) as b2:
        b.set_genome_count(G)
        for g, fa in enumerate(genomes):
            b.add_genome_bytes(g, fa)
        b.build()
        for i, g in enumerate(b_rows):
            b2.add_genome_bytes(i, genomes[g])
        rc = KmerRuleClassifications(b, G)
        pos = a_rows[labels[a_rows] == 1]
        neg = a_rows[labels[a_rows] == 0]
        _end_to_end(rc, pos, neg, b_rows, b2)


def test_predict_genomes_after_load_kover(gpu, tmp_path):
    from grm_b200 import create, hdf5min
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.learning import load_kover
    rng = np.random.default_rng(90)
    insert = inputs.rand_seq(rng, 90)
    G, k = 50, 19
    genomes, carriers = _insert_genomes(rng, G, insert)
    paths = []
    for g, fa in enumerate(genomes):
        p = tmp_path / f"g{g}.fna"
        p.write_bytes(fa)
        paths.append(str(p))
    (tmp_path / "list.tsv").write_text("".join(f"g{g}\t{p}\n" for g, p in enumerate(paths)))
    (tmp_path / "meta.tsv").write_text("".join(f"g{g}\t{int(c)}\n" for g, c in enumerate(carriers)))
    out = tmp_path / "d.kover"
    create.from_contigs(str(tmp_path / "list.tsv"), str(out), k, "nothing", "insert", str(tmp_path / "meta.tsv"), 4,
                        str(tmp_path), 2, False, False)
    r = hdf5min.H5Reader(str(out))
    ids = [int(x.decode()[1:]) for x in r["genome_identifiers"].read()]      # matrix row -> genome
    labels = r["phenotype"].read()
    rows = np.arange(len(ids))
    a_rows, b_rows = rows[np.array(ids) < 35], rows[np.array(ids) >= 35]
    with KmerMatrixBuilder(k=k) as b, KmerMatrixBuilder(k=k) as b2:
        rc = load_kover(str(out), b)
        for i, row in enumerate(b_rows):
            b2.add_genome_files(i, [paths[ids[row]]])
        _end_to_end(rc, a_rows[labels[a_rows] == 1], a_rows[labels[a_rows] == 0], b_rows, b2)
