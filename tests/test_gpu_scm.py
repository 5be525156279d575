"""The Set Covering Machine on the GPU (-m gpu): grmkm_scm_run against the numpy reference, bit for bit -- chosen
rules, utilities (as bits), counts and every set of equivalent rules -- on planted matrices, builds and .kover files."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle
from tests import inputs
from tests.scm_oracle import scm_fit

pytestmark = pytest.mark.gpu


def pack(bits):
    """(G x U) 0/1 -> (ceil(G/64) x U) uint64 words, genome g at bit 63 - g % 64 of word g // 64."""
    G, U = bits.shape
    padded = np.zeros((((G + 63) // 64) * 64, U), dtype=np.uint8)
    padded[:G] = bits
    by = np.packbits(padded.reshape(-1, 64, U).transpose(0, 2, 1), axis=2)          # (W, U, 8), big-endian
    return np.ascontiguousarray(by).view(">u8").reshape(-1, U).astype(np.uint64)


def mask(rows, G):
    m = np.zeros((G + 63) // 64, dtype=np.uint64)
    for g in rows:
        m[g // 64] |= np.uint64(1) << np.uint64(63 - g % 64)
    return m


def loaded(matrix, G):
    from grm_b200.builder import KmerMatrixBuilder
    b = KmerMatrixBuilder(k=31)
    b.load_result(np.arange(matrix.shape[1], dtype=np.uint64) * np.uint64(7919), matrix, G)
    return b


def planted(rng, G, U, n_copies=3, density=0.3):
    """Random columns, a marker column with noisy labels, and groups of identical columns (ties)."""
    bits = (rng.random((G, U)) < density).astype(np.uint8)
    marker = (rng.random(G) < 0.5).astype(np.uint8)
    labels = marker ^ (rng.random(G) < 0.1).astype(np.uint8)
    for c in rng.choice(U, size=min(U, n_copies), replace=False):
        bits[:, c] = marker
    for src in rng.choice(U, size=min(U, 8), replace=False):
        dst = rng.choice(U, size=min(U, 4), replace=False)
        bits[:, dst] = bits[:, [src]]
    return bits, labels


def same(got, want):
    steps, eq = got
    assert len(steps) == len(want)
    for s, w in zip(steps, want):
        assert int(s["rule"]) == w["rule"]
        assert np.float64(s["utility"]).view(np.int64) == np.float64(w["utility"]).view(np.int64)
        assert (int(s["positive_errors"]), int(s["negative_covers"])) == (w["positive_errors"], w["negative_covers"])
        o, n = int(s["equiv_offset"]), int(s["equiv_count"])
        assert np.array_equal(eq[o:o + n].astype(np.int64), w["equivalent"])


def run_both(b, matrix, G, pos, neg, model_type="conjunction", p=1.0, max_rules=10, blacklist=(), tiebreak=True):
    from grm_b200 import native
    mt = native.SCM_DISJUNCTION if model_type == "disjunction" else native.SCM_CONJUNCTION
    got = b.scm_run([(mt, p, max_rules, tiebreak, mask(pos, G), mask(neg, G))], np.asarray(blacklist, dtype=np.uint64))[0]
    want = scm_fit(matrix, G, pos, neg, model_type, p, max_rules, blacklist, tiebreak)
    same(got, want)
    return got, want


@pytest.mark.parametrize("G,U", [(1, 1_000_000), (63, 50_000), (64, 20_000), (65, 20_000), (300, 20_000)])
def test_planted_matrices_match_the_reference(gpu, G, U):
    rng = np.random.default_rng(G * 7 + 1)
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    pos, neg = np.nonzero(labels)[0].tolist(), np.nonzero(labels == 0)[0].tolist()
    with loaded(m, G) as b:
        for mt, p, tb in (("conjunction", 1.0, True), ("disjunction", 0.1, True), ("conjunction", 5.623, False)):
            run_both(b, m, G, pos, neg, mt, p, 10, (), tb)


def test_load_result_feeds_every_result_call(gpu):
    rng = np.random.default_rng(5)
    G, U = 130, 3000
    m = pack((rng.random((G, U)) < 0.4).astype(np.uint8))
    km = rng.integers(0, 1 << 62, size=U, dtype=np.uint64)
    from grm_b200.builder import KmerMatrixBuilder
    with KmerMatrixBuilder(k=31) as b:
        b.load_result(km, m, G)
        assert b.dims == (U, 3, G)
        assert np.array_equal(b.matrix(), m) and np.array_equal(b.kmers(), km)
        assert b.checksum() == oracle.checksum(km, m)
        rows = [0, 5, 64, 129]
        assert np.array_equal(b.sum_rows(oracle.row_mask(rows, G)), oracle.sum_rows(m, rows, G)[:U].astype(np.uint32))
        assert np.array_equal(b.gram(), oracle.gram(m, G))
        assert len(b.tsv([f"g{i}" for i in range(G)])) == 5 + sum(1 + len(f"g{i}") for i in range(G)) + 1 + U * (31 + 2 * G + 1)


@pytest.mark.parametrize("p", [0.0, 0.1, 1.0, 5.623, 999999.0])
def test_p_grid_and_edge_cases(gpu, p):
    rng = np.random.default_rng(11)
    G, U = 150, 4000
    bits, labels = planted(rng, G, U, n_copies=5)
    m = pack(bits)
    pos, neg = np.nonzero(labels)[0].tolist(), np.nonzero(labels == 0)[0].tolist()
    with loaded(m, G) as b:
        run_both(b, m, G, pos, neg, "conjunction", p)
        run_both(b, m, G, pos, neg, "disjunction", p)
        run_both(b, m, G, [], neg, "conjunction", p)                   # empty P0
        run_both(b, m, G, pos, [], "conjunction", p)                   # empty N0: no step
        # blacklist the whole best tie set of the first step: the fit must go elsewhere
        first, _ = run_both(b, m, G, pos, neg, "conjunction", p, max_rules=1, tiebreak=False)
        T = first[1][: int(first[0][0]["equiv_count"])].tolist() if len(first[0]) else []
        run_both(b, m, G, pos, neg, "conjunction", p, blacklist=T + [0, 2 * U - 1])


def test_all_negative_utilities(gpu):
    # random columns: no rule is 1 (or 0) on all 30 positives, so every rule errs on one and at p = 999999 every
    # utility is negative; the fit still takes the best of them
    rng = np.random.default_rng(12)
    G, U = 40, 500
    bits = (rng.random((G, U)) < 0.5).astype(np.uint8)
    m = pack(bits)
    with loaded(m, G) as b:
        got, want = run_both(b, m, G, list(range(0, 30)), list(range(30, 40)), "conjunction", 999999.0)
        assert want and all(w["utility"] < 0 for w in want)


def test_large_tie_set_is_complete(gpu):
    """100 000 identical columns: the tie list outgrows its first allocation and the step is redone."""
    rng = np.random.default_rng(13)
    G, U = 70, 130_000
    labels = (rng.random(G) < 0.5).astype(np.uint8)
    bits = (rng.random((G, U)) < 0.3).astype(np.uint8)
    bits[:, 20_000:120_000] = labels[:, None]
    m = pack(bits)
    pos, neg = np.nonzero(labels)[0].tolist(), np.nonzero(labels == 0)[0].tolist()
    with loaded(m, G) as b:
        got, want = run_both(b, m, G, pos, neg)
        assert len(want[0]["equivalent"]) >= 100_000


def test_batches_larger_than_one_chunk_equal_single_fits(gpu):
    """G = 32 768 (512 mask words per set): fits are chunked by shared memory; the batch equals every fit alone."""
    from grm_b200 import native
    rng = np.random.default_rng(14)
    G, U = 32768, 300
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    jobs = []
    for i in range(24):
        fold = rng.random(G) < 0.8
        pos = np.nonzero((labels == 1) & fold)[0]
        neg = np.nonzero((labels == 0) & fold)[0]
        mt = native.SCM_DISJUNCTION if i % 2 else native.SCM_CONJUNCTION
        jobs.append((mt, [0.1, 1.0, 5.623][i % 3], 3, i % 4 != 3, mask(pos, G), mask(neg, G)))
    with loaded(m, G) as b:
        batch = b.scm_run(jobs, [5, U + 7])
        for i, job in enumerate(jobs):
            alone = b.scm_run([job], [5, U + 7])[0]
            assert np.array_equal(batch[i][0], alone[0]) and np.array_equal(batch[i][1], alone[1]), i
        for i in (0, 1):
            pos = [g for g in range(G) if int(jobs[i][4][g // 64]) >> (63 - g % 64) & 1]
            neg = [g for g in range(G) if int(jobs[i][5][g // 64]) >> (63 - g % 64) & 1]
            same(batch[i], scm_fit(m, G, pos, neg, ["conjunction", "disjunction"][jobs[i][0]], jobs[i][1], 3, [5, U + 7],
                                   jobs[i][3]))


def _insert_genomes(rng, G, insert):
    core = inputs.rand_seq(rng, 4000)
    carriers = rng.random(G) < 0.5
    carriers[0], carriers[1] = True, False
    genomes = []
    for g in range(G):
        own = inputs.rand_seq(rng, 300)
        a = int(rng.integers(0, 2000))
        body = core[a:a + 1500] + own + (insert if carriers[g] else b"") + inputs.rand_seq(rng, 200)
        genomes.append(b">g%d\n" % g + body + b"\n")
    return genomes, carriers


def test_first_rule_on_a_build_is_the_insert(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.learning import KmerRuleClassifications
    from grm_b200.scm import SetCoveringMachine
    rng = np.random.default_rng(15)
    insert = inputs.rand_seq(rng, 120)
    G, k = 90, 21
    genomes, carriers = _insert_genomes(rng, G, insert)
    with KmerMatrixBuilder(k=k, keep_singletons=True) as b:
        b.set_genome_count(G)
        for g, fa in enumerate(genomes):
            b.add_genome_bytes(g, fa)
        b.build()
        U = b.dims[0]
        rc = KmerRuleClassifications(b, G)
        pos, neg = np.nonzero(carriers)[0], np.nonzero(~carriers)[0]
        m = SetCoveringMachine("conjunction", p=1.0, max_rules=5).fit(rc, pos, neg)
        want = scm_fit(b.matrix(), G, pos.tolist(), neg.tolist(), "conjunction", 1.0, 5, (), True)
        T = m.iterations[0].equivalent_rules
        assert np.array_equal(T, want[0]["equivalent"])
        assert m.iterations[0].rule == want[0]["rule"] and len(m.iterations) == len(want)
        comp = bytes.maketrans(b"ACGT", b"TGCA")
        rc_insert = insert.translate(comp)[::-1]
        strings = b.kmer_strings()
        assert (T < U).all() and len(T) > 0
        for r in T:
            s = bytes(strings[r])
            assert s in insert or s in rc_insert
        assert m.model[0].type == "presence" and m.model[0].kmer_sequence == strings[m.model[0].kmer_index].decode()
        assert m.predict(rc, pos).all()


def test_kover_round_trip(gpu, tmp_path):
    from grm_b200 import create, hdf5min
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.learning import KmerRuleClassifications, load_kover
    from grm_b200.scm import SetCoveringMachine, fit_many
    rng = np.random.default_rng(16)
    insert = inputs.rand_seq(rng, 90)
    G, k = 40, 19
    genomes, carriers = _insert_genomes(rng, G, insert)
    paths = []
    for g, fa in enumerate(genomes):
        p = tmp_path / f"g{g}.fna"
        p.write_bytes(fa)
        paths.append(str(p))
    lst = tmp_path / "list.tsv"
    lst.write_text("".join(f"g{g}\t{p}\n" for g, p in enumerate(paths)))
    meta = tmp_path / "meta.tsv"
    meta.write_text("".join(f"g{g}\t{int(c)}\n" for g, c in enumerate(carriers)))
    out = tmp_path / "d.kover"
    create.from_contigs(str(lst), str(out), k, "nothing", "insert", str(meta), 4, str(tmp_path), 2, False, False)
    r = hdf5min.H5Reader(str(out))
    ids = [int(x.decode()[1:]) for x in r["genome_identifiers"].read()]
    labels = r["phenotype"].read()
    pos, neg = np.nonzero(labels == 1)[0], np.nonzero(labels == 0)[0]

    def models(rc):
        ms = [SetCoveringMachine(t, p, 4) for t in ("conjunction", "disjunction") for p in (0.5, 1.0)]
        fit_many(rc, [(m, pos, neg) for m in ms])
        return [(m.model, [(i.rule, i.utility, i.positive_errors, i.negative_covers, i.equivalent_rules.tolist())
                           for i in m.iterations]) for m in ms]

    with KmerMatrixBuilder(k=k) as a, KmerMatrixBuilder(k=k, keep_singletons=True) as b:
        from_file = models(load_kover(str(out), a))
        b.set_genome_count(G)
        for row, g in enumerate(ids):
            b.add_genome_bytes(row, genomes[g])
        b.build()
        in_memory = models(KmerRuleClassifications(b, G))
        assert np.array_equal(a.matrix(), b.matrix()) and np.array_equal(a.kmers(), b.kmers())
    assert from_file == in_memory
    assert from_file[0][0]


def test_removed_rows_are_honoured(gpu):
    from grm_b200.learning import KmerRuleClassifications
    from grm_b200.scm import SetCoveringMachine
    rng = np.random.default_rng(17)
    G, U = 100, 5000
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    with loaded(m, G) as b:
        rc = KmerRuleClassifications(b, G)
        removed = [3, 10, 64, 99]
        rc.remove_rows(removed)
        alive = [g for g in range(G) if g not in removed]
        pos = [i for i, g in enumerate(alive) if labels[g]]
        neg = [i for i, g in enumerate(alive) if not labels[g]]
        mach = SetCoveringMachine("conjunction", 1.0, 10).fit(rc, pos, neg)
        want = scm_fit(m, G, [alive[i] for i in pos], [alive[i] for i in neg], "conjunction", 1.0, 10, (), True)
        assert [i.rule for i in mach.iterations] == [w["rule"] for w in want]
        assert all(np.array_equal(i.equivalent_rules, w["equivalent"]) for i, w in zip(mach.iterations, want))
        assert mach.predict(rc, np.arange(len(alive))).shape == (len(alive),)


def test_argument_errors(gpu):
    from grm_b200 import native
    rng = np.random.default_rng(18)
    G, U = 70, 100
    m = pack((rng.random((G, U)) < 0.5).astype(np.uint8))
    with loaded(m, G) as b:
        lib, ctx = b._lib, b._ctx

        def run(pos=None, neg=None, bl=(), **kw):
            pos = mask([0, 1], G) if pos is None else pos
            neg = mask([2, 3], G) if neg is None else neg
            f = dict(struct_size=C.sizeof(native.ScmJob), model_type=0, max_rules=3, tiebreak=1, p=1.0)
            f.update(kw)
            job = native.ScmJob(f["struct_size"], f["model_type"], f["max_rules"], f["tiebreak"], f["p"],
                                pos.ctypes.data, neg.ctypes.data)
            bl = np.asarray(bl, dtype=np.uint64)
            return lib.grmkm_scm_run(ctx, 1, C.byref(job), C.c_void_p(bl.ctypes.data), bl.size)

        assert run() == native.OK
        for kw in (dict(p=float("nan")), dict(p=-0.5), dict(p=float("inf")), dict(max_rules=0), dict(struct_size=8),
                   dict(model_type=2)):
            assert run(**kw) == native.E_INVALID, kw
        assert run(pos=mask([0], G) | np.array([0, 1], dtype=np.uint64)) == native.E_INVALID   # row 127
        assert run(neg=mask([1, 2], G)) == native.E_INVALID                                                      # overlap
        assert run(bl=[2 * U]) == native.E_INVALID
        assert run(bl=[2 * U - 1]) == native.OK
        # size query with NULL buffers
        ns, ne = C.c_uint64(), C.c_uint64()
        assert lib.grmkm_scm_result(ctx, 0, None, 0, C.byref(ns), None, 0, C.byref(ne)) in (native.E_CAPACITY, native.OK)
        assert lib.grmkm_scm_result(ctx, 1, None, 0, C.byref(ns), None, 0, C.byref(ne)) == native.E_INVALID
        bad = m.copy(); bad[1, 0] |= np.uint64(1)                   # row 127 >= G
        with pytest.raises(native.GrmkmError) as e:
            b.load_result(np.arange(U, dtype=np.uint64), bad, G)
        assert e.value.code == native.E_INVALID
        assert lib.grmkm_load_result(ctx, None, None, 0, 32769) == native.E_UNSUPPORTED


def test_a_multi_gpu_slice_is_refused(gpu):
    """An owner's slice after a two-rank merge (both ranks emulated in this process) refuses to learn."""
    import torch
    from grm_b200 import native
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import CudaEngine, row_partition, words_per_rank
    rng = np.random.default_rng(19)
    world, G = 2, 130
    genomes = [inputs.fasta(rng, n_records=2, max_len=300, shared=[inputs.rand_seq(rng, 2000)]) for _ in range(G)]
    parts, sw = row_partition(G, world), words_per_rank(G, world)
    engines = []
    for r in range(world):
        b = KmerMatrixBuilder(k=19, keep_singletons=True)
        b.set_genome_count(len(parts[r]))
        for i, g in enumerate(parts[r]):
            b.add_genome_bytes(i, genomes[g])
        engines.append(CudaEngine(b))
    bits = max(e.plan_bucket_bits() for e in engines)
    counts, sends = [], []
    for r, e in enumerate(engines):
        e.set_bucket_bits(bits)
        c, s = e.build_partial(world, sw[r])
        counts.append(c); sends.append(s)
    chunks = []
    for src in range(world):
        width = 1 + sw[src]
        chunks.append(sends[src][: counts[src][0] * width])
    engines[0].merge(torch.cat(chunks), world, 0, [counts[s][0] for s in range(world)], sw, G)
    owner = engines[0].b
    U, W, _ = owner.dims
    job = (native.SCM_CONJUNCTION, 1.0, 3, True, mask([0], G), mask([1], G))
    with pytest.raises(native.GrmkmError) as e:
        owner.scm_run([job])
    assert e.value.code == native.E_UNSUPPORTED
    owner.load_result(owner.kmers(), owner.matrix(), G)               # a whole matrix again: learning works
    owner.scm_run([job])
    for e in engines:
        e.b.close()
