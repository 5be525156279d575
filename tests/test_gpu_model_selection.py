"""Cross-validated selection on the GPU (-m gpu): grmkm_eval_run against the numpy reference, its argument checks, and
cross_validate_scm / cross_validate_cart against a brute-force composition of fit + predict with the same rules."""
import ctypes as C

import numpy as np
import pytest

from tests import inputs
from tests.eval_oracle import LEAF, eval_cart, eval_scm
from tests.test_gpu_scm import _insert_genomes, loaded, mask, pack, planted

pytestmark = pytest.mark.gpu

NO_CHILD = 0xFFFFFFFF


def random_tree(rng, U, n_max, p_split):
    """Breadth-first numbered tree of at most n_max nodes: [(kmer or LEAF, present_child, absent_child)]."""
    nodes, i = [(LEAF, 0, 0)], 0
    while i < len(nodes):
        if len(nodes) + 2 <= n_max and rng.random() < p_split:
            nodes[i] = (int(rng.integers(0, U)), len(nodes), len(nodes) + 1)
            nodes += [(LEAF, 0, 0), (LEAF, 0, 0)]
        i += 1
    return nodes


def chain_tree(rng, U, depth):
    """Every split's present child is a leaf and its absent child the next split: depth levels."""
    nodes = []
    for d in range(depth):                      # split d is node 2d, its present child (a leaf) 2d + 1
        nodes += [(int(rng.integers(0, U)), 2 * d + 1, 2 * d + 2), (LEAF, 0, 0)]
    return nodes + [(LEAF, 0, 0)]


def node_array(nodes):
    from grm_b200.builder import KmerMatrixBuilder
    return np.array([(np.iinfo(np.uint64).max, NO_CHILD, NO_CHILD) if k is LEAF else (k, p, a) for k, p, a in nodes],
                    dtype=KmerMatrixBuilder.EVAL_NODE_DTYPE)


@pytest.mark.parametrize("G", [1, 63, 64, 65, 600, 2100])
def test_eval_run_matches_the_reference(gpu, G):
    """W = 1 .. 33 words (beyond the SCM's 8 register-cached words and beyond one 32-word warp chunk), hundreds of SCM
    and tree jobs in one call: 0 rules, absence rules, both model types, single leaves, deep and wide trees, empty sets."""
    from grm_b200 import native
    rng = np.random.default_rng(G + 5)
    U = 2500
    bits = (rng.random((G, U)) < 0.4).astype(np.uint8)
    m = pack(bits)
    jobs, want = [], []
    n_jobs = 240 if G < 1000 else 80
    for i in range(n_jobs):
        x = rng.random(G)
        pos, neg = np.nonzero(x < 0.35)[0], np.nonzero((x >= 0.35) & (x < 0.7))[0]
        if i % 11 == 0:
            pos = neg = np.zeros(0, dtype=np.int64)
        elif i % 13 == 0:
            neg = np.zeros(0, dtype=np.int64)
        if i % 2 == 0:
            mt = ["conjunction", "disjunction"][(i // 2) % 2]
            rules = rng.integers(0, 2 * U, size=(i // 4) % 8).astype(np.uint64)       # 0..7 rules, half absence
            jobs.append((native.EVAL_SCM, native.SCM_DISJUNCTION if mt == "disjunction" else native.SCM_CONJUNCTION,
                         rules, mask(pos, G), mask(neg, G)))
            want.append(eval_scm(bits, mt, rules, pos, neg))
        else:
            kind = (i // 2) % 5
            nodes = ([(LEAF, 0, 0)] if kind == 0 else chain_tree(rng, U, 60) if kind == 1
                     else random_tree(rng, U, [15, 400, 3000][kind % 3], 0.8))
            jobs.append((native.EVAL_CART, 0, node_array(nodes), mask(pos, G), mask(neg, G)))
            want.append(eval_cart(bits, nodes, pos, neg))
    with loaded(m, G) as b:
        got = b.eval_run(jobs)
        assert len(got) == len(want)
        for i, (g, w) in enumerate(zip(got, want)):
            assert np.array_equal(g.astype(np.int64), w), i
        assert b.eval_run([]) == []


def test_eval_run_argument_errors(gpu):
    from grm_b200 import native
    rng = np.random.default_rng(21)
    G, U = 70, 100
    m = pack((rng.random((G, U)) < 0.5).astype(np.uint8))
    with loaded(m, G) as b:
        lib, ctx = b._lib, b._ctx
        keep = []

        def run(kind=native.EVAL_CART, rules=(), nodes=((LEAF, 0, 0),), pos=None, neg=None, cap=None, **kw):
            pos = mask([0, 1], G) if pos is None else pos
            neg = mask([2, 3], G) if neg is None else neg
            r = np.asarray(rules, dtype=np.uint64)
            nd = node_array(list(nodes))
            n = len(r) if kind == native.EVAL_SCM else len(nd)
            f = dict(struct_size=C.sizeof(native.EvalJob), kind=kind, model_type=0, reserved=0, n_items=n)
            f.update(kw)
            keep.extend([r, nd, pos, neg])
            job = native.EvalJob(f["struct_size"], f["kind"], f["model_type"], f["reserved"], f["n_items"],
                                 r.ctypes.data if len(r) else None, nd.ctypes.data if len(nd) else None,
                                 pos.ctypes.data, neg.ctypes.data)
            pairs = n + 1 if kind == native.EVAL_SCM else n
            out = np.full(2 * pairs + 2, 0xDEADBEEF, dtype=np.uint32)
            rc = lib.grmkm_eval_run(ctx, 1, C.byref(job), C.c_void_p(out.ctypes.data), 2 * pairs if cap is None else cap)
            if rc != native.OK:
                assert (out == 0xDEADBEEF).all()                # nothing written: refused before device work
            return rc

        S, T = native.EVAL_SCM, native.EVAL_CART
        assert run() == native.OK
        assert run(S, rules=[0, U, 2 * U - 1]) == native.OK
        assert run(S, rules=[]) == native.OK
        assert run(T, nodes=[(5, 1, 2), (LEAF, 0, 0), (U - 1, 3, 4), (LEAF, 0, 0), (LEAF, 0, 0)]) == native.OK
        assert run(S, rules=[2 * U]) == native.E_INVALID                               # rule >= 2U
        assert run(T, nodes=[(U, 1, 2), (LEAF, 0, 0), (LEAF, 0, 0)]) == native.E_INVALID   # k-mer >= U
        assert run(T, nodes=[(1, 1, 2), (2, 1, 3), (LEAF, 0, 0), (LEAF, 0, 0)]) == native.E_INVALID   # child <= parent
        assert run(T, nodes=[(1, 1, 3), (LEAF, 0, 0), (LEAF, 0, 0)]) == native.E_INVALID   # child >= n
        assert run(T, nodes=[(1, 1, 2), (2, 2, 3), (LEAF, 0, 0), (LEAF, 0, 0)]) == native.E_INVALID   # two parents
        assert run(T, nodes=[(1, 1, 1), (LEAF, 0, 0)]) == native.E_INVALID             # the same child twice
        assert run(T, nodes=[]) == native.E_INVALID                                    # no root
        assert run(neg=mask([1, 2], G)) == native.E_INVALID                            # overlapping masks
        assert run(pos=mask([0], G) | np.array([0, 1], dtype=np.uint64)) == native.E_INVALID   # row 127 >= G
        assert run(struct_size=8) == native.E_INVALID
        assert run(kind=2) == native.E_INVALID
        assert run(reserved=1) == native.E_INVALID
        assert run(S, model_type=2) == native.E_INVALID
        assert run(T, model_type=1) == native.E_INVALID
        assert run(S, rules=[1, 2], cap=5) == native.E_CAPACITY
        assert run(S, rules=[1, 2], pos=mask([], G), neg=mask([], G)) == native.OK      # empty masks


def test_eval_run_refuses_a_multi_gpu_slice(gpu):
    """An owner's slice after a two-rank merge (both ranks emulated in this process) refuses to evaluate."""
    import torch
    from grm_b200 import native
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import CudaEngine, row_partition, words_per_rank
    rng = np.random.default_rng(22)
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
    chunks = [sends[src][: counts[src][0] * (1 + sw[src])] for src in range(world)]
    engines[0].merge(torch.cat(chunks), world, 0, [counts[s][0] for s in range(world)], sw, G)
    owner = engines[0].b
    job = (native.EVAL_SCM, native.SCM_CONJUNCTION, [0], mask([0], G), mask([1], G))
    with pytest.raises(native.GrmkmError) as e:
        owner.eval_run([job])
    assert e.value.code == native.E_UNSUPPORTED
    owner.load_result(owner.kmers(), owner.matrix(), G)               # a whole matrix again: evaluation works
    assert owner.eval_run([job])[0].shape == (2, 2)
    for e in engines:
        e.b.close()


# -- brute-force compositions: every candidate fitted alone with `fit` and scored with `predict` ----------------------

def _errors(pred, n_pos):
    return int((pred[:n_pos] == 0).sum() + (pred[n_pos:] == 1).sum())


def brute_scm(rc, pos, neg, types, ps, R, ids):
    from grm_b200.scm import SetCoveringMachine
    pos, neg = np.asarray(pos), np.asarray(neg)
    k = int(ids.max()) + 1
    errors = np.zeros((len(types), len(ps), R), dtype=np.int64)
    for f in range(k):
        fp, fn = ids[:len(pos)] == f, ids[len(pos):] == f
        held = np.concatenate([pos[fp], neg[fn]])
        for t, mt in enumerate(types):
            for p, pv in enumerate(ps):
                mach = SetCoveringMachine(mt, pv, R).fit(rc, pos[~fp], neg[~fn])
                for r in range(1, R + 1):
                    cut = SetCoveringMachine(mt, pv, r)
                    cut.rule_indices = mach.rule_indices[:r]
                    errors[t, p, r - 1] += _errors(cut.predict(rc, held), int(fp.sum()))
    best = None
    for r in range(R):
        for t in range(len(types)):
            for p in range(len(ps)):
                if best is None or errors[t, p, r] < errors[best]:
                    best = (t, p, r)
    return errors, best


def check_scm(rc, pos, neg, types, ps, R, folds, test_pos, test_neg, seed=0):
    from grm_b200.model_selection import cross_validate_scm, make_folds
    from grm_b200.scm import SetCoveringMachine
    res = cross_validate_scm(rc, pos, neg, types, ps, R, folds, random_seed=seed, test_pos=test_pos, test_neg=test_neg)
    ids = (make_folds(np.r_[np.ones(len(pos)), np.zeros(len(neg))], folds, seed) if np.ndim(folds) == 0
           else np.asarray(folds))
    assert np.array_equal(res.fold_ids, ids)
    errors, (t, p, r) = brute_scm(rc, pos, neg, types, ps, R, ids)
    got = {(g["model_type"], g["p"], g["max_rules"]): g["cv_errors"] for g in res.grid}
    assert got == {(types[a], float(ps[b]), c + 1): int(errors[a, b, c])
                   for a in range(len(types)) for b in range(len(ps)) for c in range(R)}
    sel = res.selected
    assert (sel["model_type"], sel["p"], sel["max_rules"]) == (types[t], float(ps[p]), r + 1)
    assert sel["cv_risk"] == sel["cv_errors"] / (len(pos) + len(neg))
    fresh = SetCoveringMachine(types[t], ps[p], r + 1).fit(rc, pos, neg)
    assert res.model.max_rules == r + 1 and res.model.rule_indices == fresh.rule_indices
    assert [(i.rule, i.utility, i.positive_errors, i.negative_covers, i.equivalent_rules.tolist()) for i in res.model.iterations] == \
           [(i.rule, i.utility, i.positive_errors, i.negative_covers, i.equivalent_rules.tolist()) for i in fresh.iterations]
    for name, a, b in (("train", pos, neg), ("test", test_pos, test_neg)):
        pred = fresh.predict(rc, np.concatenate([a, b]).astype(np.int64))
        mtr = getattr(res, name)
        assert (mtr["fn"], mtr["fp"]) == (int((pred[:len(a)] == 0).sum()), int((pred[len(a):] == 1).sum())), name
    import json
    json.dumps(res.to_dict())
    return res


def brute_cart(rc, pos, neg, weights, depths, mss, ids):
    from grm_b200.cart import DecisionTreeClassifier
    pos, neg = np.asarray(pos), np.asarray(neg)
    k = int(ids.max()) + 1
    errors = np.zeros((len(weights), len(depths), len(mss)), dtype=np.int64)
    for f in range(k):
        fp, fn = ids[:len(pos)] == f, ids[len(pos):] == f
        held = np.concatenate([pos[fp], neg[fn]])
        for w, ci in enumerate(weights):
            for di, d in enumerate(depths):
                for si, s in enumerate(mss):
                    t = DecisionTreeClassifier(max_depth=d, min_samples_split=s, class_importance=ci)
                    t.fit(rc, pos[~fp], neg[~fn])
                    errors[w, di, si] += _errors(t.predict(rc, held), int(fp.sum()))
    order = sorted(((np.inf if d is None else d, -s, w, di, si) for w in range(len(weights))
                    for di, d in enumerate(depths) for si, s in enumerate(mss)))
    best = min(order, key=lambda o: (errors[o[2], o[3], o[4]], order.index(o)))
    return errors, best[2:]


def same_nodes(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert (x.rule is None) == (y.rule is None)
        if x.rule is not None:
            assert x.rule == y.rule
        assert np.float64(x.score).view(np.int64) == np.float64(y.score).view(np.int64)
        assert (x.depth, x.n_pos, x.n_neg, x.present_child, x.absent_child, x.prediction, x.equivalent_total) == \
               (y.depth, y.n_pos, y.n_neg, y.present_child, y.absent_child, y.prediction, y.equivalent_total)
        assert np.array_equal(x.equivalent_rules, y.equivalent_rules)


def check_cart(rc, pos, neg, weights, depths, mss, folds, test_pos, test_neg, seed=0):
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.model_selection import cross_validate_cart, make_folds
    res = cross_validate_cart(rc, pos, neg, weights, depths, mss, folds, random_seed=seed, test_pos=test_pos,
                              test_neg=test_neg)
    ids = (make_folds(np.r_[np.ones(len(pos)), np.zeros(len(neg))], folds, seed) if np.ndim(folds) == 0
           else np.asarray(folds))
    errors, (w, di, si) = brute_cart(rc, pos, neg, weights, depths, mss, ids)
    assert [g["cv_errors"] for g in res.grid] == errors.reshape(-1).tolist()
    sel = res.selected
    assert (sel["max_depth"], sel["min_samples_split"]) == (depths[di], mss[si])
    assert sel is res.grid[(w * len(depths) + di) * len(mss) + si]
    direct = DecisionTreeClassifier(max_depth=depths[di], min_samples_split=mss[si], class_importance=weights[w])
    direct.fit(rc, pos, neg)
    same_nodes(res.model.nodes, direct.nodes)
    assert (res.model.max_depth, res.model.min_samples_split) == (depths[di], mss[si])
    for name, a, b in (("train", pos, neg), ("test", test_pos, test_neg)):
        pred = direct.predict(rc, np.concatenate([a, b]).astype(np.int64))
        mtr = getattr(res, name)
        assert (mtr["fn"], mtr["fp"]) == (int((pred[:len(a)] == 0).sum()), int((pred[len(a):] == 1).sum())), name
        assert np.array_equal(res.model.predict(rc, np.concatenate([a, b]).astype(np.int64)), pred)
    import json
    json.dumps(res.to_dict())
    return res


def _split(rng, labels, n_test):
    idx = rng.permutation(len(labels))
    test, train = idx[:n_test], idx[n_test:]
    return ([g for g in train if labels[g]], [g for g in train if not labels[g]],
            [g for g in test if labels[g]], [g for g in test if not labels[g]])


def test_cross_validate_scm_equals_fit_and_predict(gpu):
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(23)
    G, U = 150, 4000
    bits, labels = planted(rng, G, U, density=0.4)
    labels = labels ^ (rng.random(G) < 0.15).astype(np.uint8)           # noisier: CV has something to choose
    m = pack(bits)
    pos, neg, tpos, tneg = _split(rng, labels, 30)
    with loaded(m, G) as b:
        rc = KmerRuleClassifications(b, G)
        check_scm(rc, pos, neg, ["conjunction", "disjunction"], [0.1, 1.0, 5.623], 4, 4, tpos, tneg, seed=3)


def test_cross_validate_cart_equals_fit_and_predict(gpu):
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(24)
    G, U = 150, 4000
    bits, labels = planted(rng, G, U, density=0.4)
    labels = labels ^ (rng.random(G) < 0.15).astype(np.uint8)
    m = pack(bits)
    pos, neg, tpos, tneg = _split(rng, labels, 30)
    with loaded(m, G) as b:
        rc = KmerRuleClassifications(b, G)
        check_cart(rc, pos, neg, [None, {0: 1.0, 1: 2.5}], [1, 2, 4, None], [2, 5, 12], 3, tpos, tneg, seed=4)


def test_removed_rows_and_explicit_folds(gpu):
    from grm_b200.learning import KmerRuleClassifications
    rng = np.random.default_rng(25)
    G, U = 100, 3000
    bits, labels = planted(rng, G, U, density=0.4)
    m = pack(bits)
    with loaded(m, G) as b:
        rc = KmerRuleClassifications(b, G)
        removed = [3, 10, 64, 99]
        rc.remove_rows(removed)
        alive = np.array([g for g in range(G) if g not in removed])
        lab = labels[alive]
        pos, neg, tpos, tneg = _split(rng, lab, 20)
        ids = np.arange(len(pos) + len(neg)) % 3                        # e.g. lineage groups, not stratified
        check_scm(rc, pos, neg, ["conjunction"], [1.0, 0.316], 3, ids, tpos, tneg)
        check_cart(rc, pos, neg, [None], [1, 3], [2, 10], ids, tpos, tneg)


def test_a_planted_rule_is_selected_with_zero_cv_error(gpu):
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.learning import KmerRuleClassifications
    from grm_b200.model_selection import cross_validate_cart, cross_validate_scm
    rng = np.random.default_rng(26)
    insert = inputs.rand_seq(rng, 120)
    G, k = 90, 21
    genomes, carriers = _insert_genomes(rng, G, insert)
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    rc_insert = insert.translate(comp)[::-1]
    with KmerMatrixBuilder(k=k, keep_singletons=True) as b:
        b.set_genome_count(G)
        for g, fa in enumerate(genomes):
            b.add_genome_bytes(g, fa)
        b.build()
        rc = KmerRuleClassifications(b, G)
        pos, neg = np.nonzero(carriers)[0], np.nonzero(~carriers)[0]
        res = cross_validate_scm(rc, pos, neg, ["conjunction", "disjunction"], [1.0, 10.0], 3, 5)
        assert res.selected["cv_errors"] == 0 and res.selected["max_rules"] == 1
        assert res.selected["model_type"] == "conjunction" and res.train["risk"] == 0
        s = res.model.model[0].kmer_sequence.encode()
        assert res.model.model[0].type == "presence" and (s in insert or s in rc_insert)
        res = cross_validate_cart(rc, pos, neg, [None], [1, 2, 3], [2], 5)
        assert res.selected["cv_errors"] == 0 and res.selected["max_depth"] == 1
        s = res.model.nodes[0].rule.kmer_sequence.encode()
        assert len(res.model.nodes) == 3 and (s in insert or s in rc_insert)
