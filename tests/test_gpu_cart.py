"""CART on the GPU (-m gpu): grmkm_cart_run against the numpy reference, bit for bit -- node order, rules, scores (as
bits), counts, children, predictions, recorded equivalent rules and their totals -- on planted matrices, builds and
.kover files."""
import numpy as np
import pytest

from tests import inputs
from tests.cart_oracle import LEAF, cart_fit, cart_predict
from tests.test_gpu_scm import _insert_genomes, loaded, mask, pack, planted

pytestmark = pytest.mark.gpu

UNLIMITED = 2**32 - 1
ALL = 2**64 - 1


def same(got, want):
    nodes, eq = got
    assert len(nodes) == len(want)
    for i, (n, w) in enumerate(zip(nodes, want)):
        leaf = w["rule"] == LEAF
        assert int(n["rule"]) == (2**64 - 1 if leaf else w["rule"]), i
        assert np.float64(n["score"]).view(np.int64) == np.float64(w["score"]).view(np.int64), i
        assert (int(n["depth"]), int(n["n_pos"]), int(n["n_neg"]), int(n["prediction"])) == \
               (w["depth"], w["n_pos"], w["n_neg"], w["prediction"]), i
        assert int(n["present_child"]) == (UNLIMITED if leaf else w["present_child"]), i
        assert int(n["absent_child"]) == (UNLIMITED if leaf else w["absent_child"]), i
        o, c = int(n["equiv_offset"]), int(n["equiv_count"])
        assert np.array_equal(eq[o:o + c].astype(np.int64), w["equivalent"]), i
        assert int(n["equiv_total"]) == w["equiv_total"], i


def job(G, pos, neg, max_depth=None, min_samples_split=2, equiv_cap=None, w_neg=1.0, w_pos=1.0):
    return (UNLIMITED if max_depth is None else max_depth, min_samples_split, ALL if equiv_cap is None else equiv_cap,
            w_neg, w_pos, mask(pos, G), mask(neg, G))


def run_both(b, matrix, G, pos, neg, blacklist=(), **kw):
    got = b.cart_run([job(G, pos, neg, **kw)], np.asarray(blacklist, dtype=np.uint64))[0]
    want = cart_fit(matrix, G, pos, neg, blacklist=blacklist, **kw)
    same(got, want)
    return got, want


def rows(labels):
    return np.nonzero(labels)[0].tolist(), np.nonzero(labels == 0)[0].tolist()


@pytest.mark.parametrize("G,U", [(1, 1_000_000), (2, 200_000), (63, 50_000), (64, 20_000), (65, 20_000),
                                 (300, 20_000)])
def test_planted_matrices_match_the_reference(gpu, G, U):
    rng = np.random.default_rng(G * 5 + 3)
    bits, labels = planted(rng, G, U)
    if G == 2:
        labels = np.array([1, 0], dtype=np.uint8)
    m = pack(bits)
    pos, neg = rows(labels)
    with loaded(m, G) as b:
        run_both(b, m, G, pos, neg)                                                      # until pure
        run_both(b, m, G, pos, neg, max_depth=1)
        run_both(b, m, G, pos, neg, max_depth=3, min_samples_split=5, w_neg=0.7, w_pos=2.5, blacklist=[1, U + 3])
        run_both(b, m, G, pos, neg, min_samples_split=5, w_neg=3.0, w_pos=0.25, equiv_cap=3)


def test_blacklisting_the_best_tie_set(gpu):
    rng = np.random.default_rng(21)
    G, U = 150, 4000
    bits, labels = planted(rng, G, U, n_copies=5)
    m = pack(bits)
    pos, neg = rows(labels)
    with loaded(m, G) as b:
        first, want = run_both(b, m, G, pos, neg, max_depth=1)
        T = want[0]["equivalent"].tolist()
        assert len(T) >= 5                                    # the planted marker copies
        # either twin of every member removes it: the root must split elsewhere
        bl = [j if i % 2 else U + j for i, j in enumerate(T)]
        _, again = run_both(b, m, G, pos, neg, blacklist=bl, max_depth=3)
        assert again[0]["rule"] not in T


def test_empty_example_sets(gpu):
    rng = np.random.default_rng(22)
    G, U = 100, 3000
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    pos, neg = rows(labels)
    with loaded(m, G) as b:
        got = b.cart_run([job(G, [], []), job(G, pos, []), job(G, [], neg), job(G, pos, neg, max_depth=2)])
        for (nodes, eq), (p, n) in zip(got, [([], []), (pos, []), ([], neg), (pos, neg)]):
            same((nodes, eq), cart_fit(m, G, p, n, max_depth=2))
        assert [len(x[0]) for x in got[:3]] == [1, 1, 1]


def test_large_tie_set_is_complete_or_capped(gpu):
    """100 000 identical perfectly splitting columns: uncapped, the tie list outgrows its first allocation and the
    level is redone; with equiv_cap = 10 the node records the 10 smallest members and the total."""
    rng = np.random.default_rng(23)
    G, U = 70, 130_000
    labels = (rng.random(G) < 0.5).astype(np.uint8)
    bits = (rng.random((G, U)) < 0.3).astype(np.uint8)
    bits[:, 20_000:120_000] = labels[:, None]
    m = pack(bits)
    pos, neg = rows(labels)
    with loaded(m, G) as b:
        got, want = run_both(b, m, G, pos, neg)
        assert want[0]["equiv_total"] >= 100_000 and len(want[0]["equivalent"]) == want[0]["equiv_total"]
        got, want = run_both(b, m, G, pos, neg, equiv_cap=10)
        assert int(got[0][0]["equiv_count"]) == 10 and int(got[0][0]["equiv_total"]) >= 100_000


def test_deep_ties_with_a_small_cap_stay_in_bounded_memory(gpu):
    """Grown until pure on 64 genomes: the bottom nodes (one positive, one negative) tie on every column that tells
    them apart, about half of 10^6 columns each.  With equiv_cap = 4 the tie list stays near 4 + one CTA's columns
    per node."""
    rng = np.random.default_rng(24)
    G, U = 64, 1_000_000
    bits = (rng.random((G, U)) < 0.5).astype(np.uint8)
    labels = (rng.random(G) < 0.5).astype(np.uint8)
    m = pack(bits)
    pos, neg = rows(labels)
    with loaded(m, G) as b:
        before = b.stats["device_bytes"]
        got, want = run_both(b, m, G, pos, neg, equiv_cap=4)
        grown = b.stats["device_bytes"] - before
        assert max(w["equiv_total"] for w in want) > 100_000
        every_tie = sum(w["equiv_total"] for w in want) * 8
        assert grown < 32 << 20 and grown < every_tie // 4, (grown, every_tie)


def test_levels_wider_than_one_chunk_equal_single_trees(gpu):
    """G = 32 768 (512 mask words per set): a level of many open nodes spans several shared-memory chunks; the batch
    equals every tree fitted alone, and two trees equal the reference."""
    rng = np.random.default_rng(25)
    G, U = 32768, 300
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    jobs, sets = [], []
    for i in range(8):
        fold = rng.random(G) < 0.8
        pos, neg = np.nonzero((labels == 1) & fold)[0], np.nonzero((labels == 0) & fold)[0]
        sets.append((pos, neg))
        jobs.append(job(G, pos, neg, max_depth=4, min_samples_split=[2, 5][i % 2], equiv_cap=[None, 3][i % 2],
                        w_neg=[1.0, 0.5][i % 2], w_pos=1.0))
    bl = [5, U + 7]
    with loaded(m, G) as b:
        batch = b.cart_run(jobs, bl)
        assert sum(int((x[0]["depth"] == 2).sum()) for x in batch) > 7          # the chunk holds 7 nodes at W = 512
        for i, j in enumerate(jobs):
            alone = b.cart_run([j], bl)[0]
            assert np.array_equal(batch[i][0], alone[0]) and np.array_equal(batch[i][1], alone[1]), i
        for i in (0, 1):
            pos, neg = sets[i]
            same(batch[i], cart_fit(m, G, pos.tolist(), neg.tolist(), 4, [2, 5][i], [1.0, 0.5][i], 1.0, bl, [None, 3][i]))


def test_truncation_property(gpu):
    rng = np.random.default_rng(26)
    G, U = 200, 20_000
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    pos, neg = rows(labels)
    with loaded(m, G) as b:
        out = b.cart_run([job(G, pos, neg)] + [job(G, pos, neg, max_depth=d) for d in (1, 2, 3)])
        full = out[0][0]
        assert int(full["depth"].max()) > 3
        for d, (cut, _) in zip((1, 2, 3), out[1:]):
            keep = full[full["depth"] <= d]
            assert len(cut) == len(keep)
            for f in ("n_pos", "n_neg", "depth", "equiv_total", "prediction"):
                assert np.array_equal(cut[f][cut["depth"] < d], keep[f][keep["depth"] < d]), f
            assert np.array_equal(cut["rule"][cut["depth"] < d], keep["rule"][keep["depth"] < d])
            assert (cut["rule"][cut["depth"] == d] == 2**64 - 1).all()


def test_predict_matches_the_reference_tree(gpu):
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(27)
    G, U = 160, 8000
    bits, labels = planted(rng, G, U)
    m = pack(bits)
    train = rng.random(G) < 0.7
    pos, neg = np.nonzero(train & (labels == 1))[0], np.nonzero(train & (labels == 0))[0]
    with loaded(m, G) as b:
        rc = KmerRuleClassifications(b, G)
        t = DecisionTreeClassifier(max_depth=4, class_importance={0: 1.0, 1: 1.5}).fit(rc, pos, neg)
        want = cart_fit(m, G, pos.tolist(), neg.tolist(), 4, 2, 1.0, 1.5)
        assert [(-1 if x.rule is None else x.rule.kmer_index) for x in t.nodes] == [w["rule"] for w in want]
        everyone = np.arange(G)
        assert np.array_equal(t.predict(rc, everyone), cart_predict(want, m, G, everyone))


def test_root_split_on_a_build_is_the_insert(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(28)
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
        t = DecisionTreeClassifier(max_depth=3).fit(rc, pos, neg)
        want = cart_fit(b.matrix(), G, pos.tolist(), neg.tolist(), 3)
        root = t.nodes[0]
        assert root.score == 0.0 and np.array_equal(root.equivalent_rules, want[0]["equivalent"])
        assert root.equivalent_total == len(root.equivalent_rules) > 0
        comp = bytes.maketrans(b"ACGT", b"TGCA")
        rc_insert = insert.translate(comp)[::-1]
        strings = b.kmer_strings()
        assert (root.equivalent_rules < U).all()
        for j in root.equivalent_rules:
            s = bytes(strings[j])
            assert s in insert or s in rc_insert
        assert root.rule.kmer_index == want[0]["rule"] and root.rule.kmer_sequence == strings[root.rule.kmer_index].decode()
        assert len(t.nodes) == 3 and np.array_equal(t.predict(rc, np.arange(G)), carriers.astype(np.uint8))


def test_kover_round_trip(gpu, tmp_path):
    from grm_b200 import create, hdf5min
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.cart import DecisionTreeClassifier, fit_many
    from grm_b200.learning import KmerRuleClassifications, load_kover
    rng = np.random.default_rng(29)
    insert = inputs.rand_seq(rng, 90)
    G, k = 40, 19
    genomes, carriers = _insert_genomes(rng, G, insert)
    carriers[2:6] = ~carriers[2:6]                # label noise: the trees need more than one split
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

    def trees(rc):
        ts = [DecisionTreeClassifier(max_depth=d, class_importance=ci, max_equivalent_rules=50)
              for d in (2, None) for ci in (None, {0: 2.0, 1: 1.0})]
        fit_many(rc, [(t, pos, neg) for t in ts])
        return [[(x.rule, x.score, x.n_pos, x.n_neg, x.present_child, x.absent_child, x.prediction,
                  x.equivalent_rules.tolist(), x.equivalent_total) for x in t.nodes] for t in ts]

    with KmerMatrixBuilder(k=k) as a, KmerMatrixBuilder(k=k, keep_singletons=True) as b:
        from_file = trees(load_kover(str(out), a))
        b.set_genome_count(G)
        for row, g in enumerate(ids):
            b.add_genome_bytes(row, genomes[g])
        b.build()
        in_memory = trees(KmerRuleClassifications(b, G))
        assert np.array_equal(a.matrix(), b.matrix()) and np.array_equal(a.kmers(), b.kmers())
        same(b.cart_run([job(G, pos, neg, max_depth=2, equiv_cap=50)])[0],
             cart_fit(b.matrix(), G, pos.tolist(), neg.tolist(), 2, equiv_cap=50))
    assert from_file == in_memory
    assert len(from_file[2]) > 3


def test_removed_rows_are_honoured(gpu):
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(30)
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
        t = DecisionTreeClassifier(max_depth=None).fit(rc, pos, neg)
        want = cart_fit(m, G, [alive[i] for i in pos], [alive[i] for i in neg], None)
        assert [(-1 if x.rule is None else x.rule.kmer_index) for x in t.nodes] == [w["rule"] for w in want]
        assert all(np.array_equal(x.equivalent_rules, w["equivalent"]) for x, w in zip(t.nodes, want))
        assert np.array_equal(t.predict(rc, np.arange(len(alive))), cart_predict(want, m, G, alive))


def test_argument_errors(gpu):
    import ctypes as C
    from grm_b200 import native
    rng = np.random.default_rng(31)
    G, U = 70, 100
    m = pack((rng.random((G, U)) < 0.5).astype(np.uint8))
    with loaded(m, G) as b:
        lib, ctx = b._lib, b._ctx

        def run(pos=None, neg=None, bl=(), **kw):
            pos = mask([0, 1], G) if pos is None else pos
            neg = mask([2, 3], G) if neg is None else neg
            f = dict(struct_size=C.sizeof(native.CartJob), max_depth=3, min_samples_split=2, reserved=0, equiv_cap=5,
                     w_neg=1.0, w_pos=1.0)
            f.update(kw)
            j = native.CartJob(f["struct_size"], f["max_depth"], f["min_samples_split"], f["reserved"], f["equiv_cap"],
                               f["w_neg"], f["w_pos"], pos.ctypes.data, neg.ctypes.data)
            bl = np.asarray(bl, dtype=np.uint64)
            return lib.grmkm_cart_run(ctx, 1, C.byref(j), C.c_void_p(bl.ctypes.data), bl.size)

        assert run() == native.OK
        for kw in (dict(struct_size=8), dict(max_depth=0), dict(min_samples_split=1), dict(reserved=1),
                   dict(w_neg=0.0), dict(w_pos=-1.0), dict(w_pos=float("nan")), dict(w_neg=float("inf")),
                   dict(w_pos=1e101)):
            assert run(**kw) == native.E_INVALID, kw
        assert run(pos=mask([0], G) | np.array([0, 1], dtype=np.uint64)) == native.E_INVALID     # row 127
        assert run(neg=mask([1, 2], G)) == native.E_INVALID                                       # overlap
        assert run(bl=[2 * U]) == native.E_INVALID
        assert run(bl=[2 * U - 1]) == native.OK
        nn, ne = C.c_uint64(), C.c_uint64()
        assert lib.grmkm_cart_result(ctx, 0, None, 0, C.byref(nn), None, 0, C.byref(ne)) in (native.E_CAPACITY, native.OK)
        assert nn.value >= 1
        assert lib.grmkm_cart_result(ctx, 1, None, 0, C.byref(nn), None, 0, C.byref(ne)) == native.E_INVALID
        b.load_result(np.arange(U, dtype=np.uint64), m, G)          # a new result forgets the trees
        assert lib.grmkm_cart_result(ctx, 0, None, 0, C.byref(nn), None, 0, C.byref(ne)) == native.E_INVALID
