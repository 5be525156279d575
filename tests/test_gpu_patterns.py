"""Distinct presence patterns (-m gpu): grmkm_patterns against the numpy reference (tests/pattern_oracle.py), and the
learners on a PatternRuleClassifications bit for bit equal to the same calls on the whole matrix -- SCM grids, CART
trees with capped and complete tie lists, both CV selections, predict, get_columns and sum_rows."""
import json

import numpy as np
import pytest

from tests import inputs
from tests.pattern_oracle import reference_patterns
from tests.test_gpu_scm import loaded, pack, planted

pytestmark = pytest.mark.gpu


def check_patterns(b, m, G, column_class=None):
    """b.patterns into a second builder equals the reference; the second builder holds the head columns."""
    from grm_b200.builder import KmerMatrixBuilder
    want = reference_patterns(m, column_class)
    with KmerMatrixBuilder(k=31) as dst:
        pattern_of, members, offsets, st = b.patterns(dst, column_class, with_stats=True)
        assert np.array_equal(pattern_of, want[0])
        assert np.array_equal(members, want[1])
        assert np.array_equal(offsets, want[2])
        P = len(want[2]) - 1
        heads = want[1][want[2][:-1]]
        assert st["n_patterns"] == P and st["n_rounds"] >= (1 if m.shape[1] else 0)
        assert dst.dims == (P, m.shape[0], G)
        assert np.array_equal(dst.matrix(), m[:, heads])
        assert np.array_equal(dst.kmers(), b.kmers()[heads])
        return st


def duplicated(rng, G, U, n_base, density=0.3):
    base = (rng.random((G, n_base)) < density).astype(np.uint8)
    return base[:, rng.integers(0, n_base, size=U)]


@pytest.mark.parametrize("G", [1, 63, 64, 65, 300])
def test_patterns_match_the_reference(gpu, G):
    rng = np.random.default_rng(G)
    cases = [duplicated(rng, G, 5000, 300),                        # many members per pattern
             (rng.random((G, 3000)) < 0.5).astype(np.uint8),       # all distinct unless G is small
             np.ones((G, 2000), dtype=np.uint8),                   # one pattern of U members
             np.zeros((G, 255), dtype=np.uint8), duplicated(rng, G, 256, 40), duplicated(rng, G, 257, 40)]
    for bits in cases:
        m = pack(bits)
        with loaded(m, G) as b:
            check_patterns(b, m, G)
            cls = rng.integers(0, 4, size=m.shape[1]).astype(np.uint8)        # class splits
            check_patterns(b, m, G, cls)


def test_zero_columns_and_a_million(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    with KmerMatrixBuilder(k=31) as b:
        b.load_result(np.zeros(0, dtype=np.uint64), np.zeros((2, 0), dtype=np.uint64), 65)
        check_patterns(b, np.zeros((2, 0), dtype=np.uint64), 65)
    rng = np.random.default_rng(7)
    G, U = 65, 1_000_000
    m = pack(duplicated(rng, G, U, 20000))
    with loaded(m, G) as b:
        st = check_patterns(b, m, G)
    assert st["n_rounds"] == 1


def test_truncated_fingerprints_force_rounds(gpu, monkeypatch):
    rng = np.random.default_rng(11)
    G = 65
    m = pack(duplicated(rng, G, 20000, 500))
    cls = (rng.random(m.shape[1]) < 0.2).astype(np.uint8) * 3
    with loaded(m, G) as b:
        for bits in ("1", "3", "8"):
            monkeypatch.setenv("GRMKM_PATTERN_HASH_BITS", bits)
            st = check_patterns(b, m, G)
            assert st["n_rounds"] > 1
            check_patterns(b, m, G, cls)


def test_patterns_of_a_build(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(3)
    shared = [inputs.rand_seq(rng, 3000), inputs.rand_seq(rng, 1500)]
    G = 70
    with KmerMatrixBuilder(k=21) as b:
        for g in range(G):
            b.add_genome_bytes(g, inputs.fasta(rng, n_records=2, max_len=400, shared=shared))
        b.build()
        m = b.matrix()
        st = check_patterns(b, m, G)
        assert st["n_patterns"] * 5 < m.shape[1]


def both(m, G, blacklist=None):
    """(whole-matrix rc, view) of the same matrix."""
    from grm_b200.learning import KmerRuleClassifications, PatternRuleClassifications
    b = loaded(m, G)
    rc = KmerRuleClassifications(b, G)
    return rc, PatternRuleClassifications(rc, blacklist)


def iterations_equal(a, b):
    assert a.rule_indices == b.rule_indices and a.model == b.model
    assert len(a.iterations) == len(b.iterations)
    for x, y in zip(a.iterations, b.iterations):
        assert (x.rule, x.positive_errors, x.negative_covers) == (y.rule, y.positive_errors, y.negative_covers)
        assert np.float64(x.utility).view(np.int64) == np.float64(y.utility).view(np.int64)
        assert np.array_equal(x.equivalent_rules, y.equivalent_rules)


@pytest.mark.parametrize("G", [1, 64, 65, 300])
def test_scm_grid_on_the_view_equals_the_whole_matrix(gpu, G):
    from grm_b200 import scm
    rng = np.random.default_rng(50 + G)
    U = 4000
    bits, labels = planted(rng, G, U, n_copies=6)
    bits[:, 2000:2400] = bits[:, rng.integers(0, 2000, size=400)]        # many multi-member patterns
    m = pack(bits)
    bl = [int(x) for x in rng.choice(U, size=10, replace=False)]
    bl += [U + int(x) for x in rng.choice(U, size=10, replace=False)]
    bl += [2000, U + 2001]                                               # one member of a pattern, not the others
    rc, view = both(m, G, bl)
    assert view.n_patterns < U
    fits = [[], []]
    for f in range(10):
        sub = rng.random(G) < 0.8
        pos = [g for g in range(G) if labels[g] and sub[g]]
        neg = [g for g in range(G) if not labels[g] and sub[g]]
        for mt in ("conjunction", "disjunction"):
            for p in (0.1, 0.5, 1.0, 2.0, 5.0, 10.0):
                for i in range(2):
                    fits[i].append((scm.SetCoveringMachine(mt, p, 6), pos, neg))
    assert len(fits[0]) == 120
    for tb in ("risk", None):
        scm.fit_many(rc, fits[0], bl, tb)
        scm.fit_many(view, fits[1], list(reversed(bl)), tb)
        for (a, _, _), (b, _, _) in zip(*fits):
            iterations_equal(a, b)
    view.close()
    rc.builder.close()


@pytest.mark.parametrize("G", [63, 300])
def test_cart_on_the_view_equals_the_whole_matrix(gpu, G):
    from grm_b200.cart import DecisionTreeClassifier, fit_many
    rng = np.random.default_rng(70 + G)
    U = 3000
    bits, labels = planted(rng, G, U, n_copies=5)
    bits[:, 1500:1600] = bits[:, [3]]
    m = pack(bits)
    pos = [g for g in range(G) if labels[g]]
    neg = [g for g in range(G) if not labels[g]]
    bl = [1550, U + 7]
    rc, view = both(m, G, bl)
    trees = [[], []]
    for cap in (None, 1, 10, 0):
        for ci in (None, {0: 0.3, 1: 2.0}):
            for mss in (2, 7):
                for i in range(2):
                    trees[i].append((DecisionTreeClassifier("gini", 6, mss, ci, cap), pos, neg))
    fit_many(rc, trees[0], bl)
    fit_many(view, trees[1], bl)
    for (a, _, _), (b, _, _) in zip(*trees):
        assert str(a.nodes) == str(b.nodes)
    view.close()
    rc.builder.close()


def test_a_single_pattern_tie_of_100000_members(gpu):
    """100 000 copies of the label column: one pattern, one tie set; equivalent_total is exact and the list capped."""
    from grm_b200.cart import DecisionTreeClassifier
    rng = np.random.default_rng(13)
    G, U = 130, 120_000
    labels = (rng.random(G) < 0.5).astype(np.uint8)
    bits = (rng.random((G, U)) < 0.3).astype(np.uint8)
    cols = np.sort(rng.choice(U, size=100_000, replace=False))
    bits[:, cols] = labels[:, None]
    m = pack(bits)
    pos, neg = np.nonzero(labels)[0], np.nonzero(labels == 0)[0]
    rc, view = both(m, G)
    for cap in (None, 1, 10):
        a = DecisionTreeClassifier(max_depth=2, max_equivalent_rules=cap).fit(rc, pos, neg)
        b = DecisionTreeClassifier(max_depth=2, max_equivalent_rules=cap).fit(view, pos, neg)
        assert str(a.nodes) == str(b.nodes)
        assert b.nodes[0].equivalent_total == 100_000
        assert np.array_equal(b.nodes[0].equivalent_rules, cols[: 100_000 if cap is None else cap])
    view.close()
    rc.builder.close()


def selection_json(res):
    d = res.to_dict()
    d.pop("seconds")
    return json.dumps(d, sort_keys=True)


def test_cross_validation_predict_columns_and_sums_on_the_view(gpu):
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.model_selection import cross_validate_cart, cross_validate_scm
    from grm_b200.scm import SetCoveringMachine
    rng = np.random.default_rng(41)
    G, U = 150, 6000
    bits, labels = planted(rng, G, U, density=0.4)
    bits[:, 3000:] = bits[:, rng.integers(0, 3000, size=U - 3000)]
    labels = labels ^ (rng.random(G) < 0.15).astype(np.uint8)
    m = pack(bits)
    alive = G - 2                                       # rows 7 and 8 are removed: example indices count the others
    pos = [g for g in range(115) if labels[g]]
    neg = [g for g in range(115) if not labels[g]]
    tpos = [g for g in range(115, alive) if labels[g]]
    tneg = [g for g in range(115, alive) if not labels[g]]
    bl = [5, U + 3100]

    def run(rc):
        rc.remove_rows([7, 8])
        a = cross_validate_scm(rc, pos, neg, ["conjunction", "disjunction"], [0.1, 1.0, 5.6], 4, 4, test_pos=tpos,
                               test_neg=tneg, random_seed=3, rule_blacklist=bl)
        b = cross_validate_cart(rc, pos, neg, [{0: 1.0, 1: 1.0}, {0: 0.5, 1: 2.0}], [1, 2, 4], [2, 10], 3,
                                test_pos=tpos, test_neg=tneg, max_equivalent_rules=5, rule_blacklist=bl)
        s = SetCoveringMachine("disjunction", 1.0, 5).fit(rc, pos, neg, bl)
        t = DecisionTreeClassifier(max_depth=4, max_equivalent_rules=3).fit(rc, pos, neg, bl)
        test = tpos[:-2] + tneg[:-2]
        return (selection_json(a), selection_json(b), s.model, s.predict(rc, test), str(t.nodes), t.predict(rc, test),
                rc.get_columns([5, 3001, U + 7, U + 3500]), rc.get_columns(4000), rc.sum_rows(test))

    rc, view = both(m, G, bl)
    want, got = run(rc), run(view)
    assert got[:3] == want[:3] and got[4] == want[4]
    for i in (3, 5, 6, 7, 8):
        assert np.array_equal(got[i], want[i]), i
    view.close()
    rc.builder.close()


def test_refusals(gpu):
    from grm_b200 import native
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import ThreadExchange
    from grm_b200.learning import PatternRuleClassifications, ShardedRuleClassifications
    from grm_b200.scm import SetCoveringMachine
    rng = np.random.default_rng(2)
    G, U = 70, 500
    m = pack((rng.random((G, U)) < 0.3).astype(np.uint8))
    with loaded(m, G) as b, KmerMatrixBuilder(k=31) as dst, KmerMatrixBuilder(k=31) as empty:
        with pytest.raises(native.GrmkmError) as e:
            b.patterns(b)
        assert e.value.code == native.E_INVALID
        with pytest.raises(native.GrmkmError) as e:
            b.patterns(dst, np.full(U, 4, dtype=np.uint8))
        assert e.value.code == native.E_INVALID and "> 3" in str(e.value)
        with pytest.raises(native.GrmkmError) as e:
            empty.patterns(dst)
        assert e.value.code == native.E_INVALID
        rc = ShardedRuleClassifications(b, G, 0, 1, [U], ThreadExchange.group(1)[0])
        with pytest.raises(ValueError):
            PatternRuleClassifications(rc)
        from grm_b200.learning import KmerRuleClassifications
        view = PatternRuleClassifications(KmerRuleClassifications(b, G), [3, U + 4])
        with pytest.raises(ValueError, match="build a PatternRuleClassifications"):
            SetCoveringMachine().fit(view, [0, 1, 2], [3, 4, 5], [3])
        SetCoveringMachine().fit(view, [0, 1, 2], [3, 4, 5], [U + 4, 3])
        view.close()
    # a multi-GPU owner slice: the merge of two partial builds emulated in this process
    import torch
    from grm_b200.distributed import CudaEngine, row_partition, words_per_rank
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
    with KmerMatrixBuilder(k=19) as dst:
        with pytest.raises(native.GrmkmError) as e:
            engines[0].b.patterns(dst)
        assert e.value.code == native.E_UNSUPPORTED
    for e in engines:
        e.b.close()
