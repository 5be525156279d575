"""CPU: the CART numpy reference on hand-computed cases, the layouts of the new ABI structs, and the argument errors
that need no device."""
import ctypes as C

import numpy as np
import pytest

import tests.test_scm_cpu as scm_cpu
from grm_b200 import native
from tests.cart_oracle import LEAF, cart_fit, cart_predict

# genomes g0..g3 (rows) x k-mers k0..k4 (columns); positives g0, g1, negatives g2, g3
BITS = np.array([[0, 1, 0, 1, 1],
                 [1, 1, 0, 1, 0],
                 [0, 0, 1, 1, 0],
                 [1, 0, 1, 1, 0]])


def tree(bits=BITS, pos=(0, 1), neg=(2, 3), **kw):
    nodes = cart_fit(scm_cpu.packed(bits), bits.shape[0], list(pos), list(neg), **kw)
    return [(n["rule"], n["score"], n["depth"], n["n_pos"], n["n_neg"], n["present_child"], n["absent_child"],
             n["prediction"], n["equivalent"].tolist(), n["equiv_total"]) for n in nodes]


def test_perfect_split_and_tie_resolved_by_min_index():
    # k1 (present on both positives only) and k2 (on both negatives only) split perfectly: score 0 + 0.  k0: two
    # (1, 1) children, 1/2 + 1/2 = 1; k4: (1, 0) and (1, 2), 0 + 2/3; k3 is on every genome (empty absent child)
    assert tree() == [(1, 0.0, 0, 2, 2, 1, 2, 0, [1, 2], 2),
                      (LEAF, 0.0, 1, 2, 0, LEAF, LEAF, 1, [], 0),
                      (LEAF, 0.0, 1, 0, 2, LEAF, LEAF, 0, [], 0)]


def test_blacklist_either_twin_removes_the_kmer():
    assert tree(blacklist=[1])[0][0] == 2 and tree(blacklist=[5 + 1])[0][0] == 2
    assert tree(blacklist=[1])[0][8] == [2]


def test_deeper_tree_breadth_first():
    # without k1 and k2: k4 (0 + 2/3) beats k0 (1/2 + 1/2).  Its absent child {g1 +, g2 -, g3 -} splits on k0:
    # {g1, g3} (1, 1) -> 1/2, {g2} -> 0.  {g1, g3} is left with no admissible split (k0, k3 on both, k4 on neither): a
    # leaf, and A == B == 1 predicts 0
    assert tree(blacklist=[1, 2]) == [(4, 2 / 3, 0, 2, 2, 1, 2, 0, [4], 1),
                                      (LEAF, 0.0, 1, 1, 0, LEAF, LEAF, 1, [], 0),
                                      (0, 0.5, 1, 1, 2, 3, 4, 0, [0], 1),
                                      (LEAF, 0.0, 2, 1, 1, LEAF, LEAF, 0, [], 0),
                                      (LEAF, 0.0, 2, 0, 1, LEAF, LEAF, 0, [], 0)]


def test_stop_rules():
    # max_depth 1: only the root splits
    got = tree(blacklist=[1, 2], max_depth=1)
    assert [n[0] for n in got] == [4, LEAF, LEAF]
    assert [(n[3], n[4], n[7]) for n in got] == [(2, 2, 0), (1, 0, 1), (1, 2, 0)]
    # min_samples_split 4: the absent child (3 examples) is a leaf -- the same tree
    assert tree(blacklist=[1, 2], min_samples_split=4) == got
    # min_samples_split 5: the root (4 examples) is a leaf; A == B == 2 predicts 0
    assert tree(blacklist=[1, 2], min_samples_split=5) == [(LEAF, 0.0, 0, 2, 2, LEAF, LEAF, 0, [], 0)]


def test_pure_node_and_empty_sets_are_leaves():
    assert tree(neg=()) == [(LEAF, 0.0, 0, 2, 0, LEAF, LEAF, 1, [], 0)]
    assert tree(pos=(), neg=()) == [(LEAF, 0.0, 0, 0, 0, LEAF, LEAF, 0, [], 0)]


def test_no_admissible_split_is_a_leaf():
    # only k3 (on every genome) is left
    assert tree(blacklist=[0, 1, 2, 4]) == [(LEAF, 0.0, 0, 2, 2, LEAF, LEAF, 0, [], 0)]


# g0..g2 positive, g3..g5 negative; Y (k0) sends g0 alone to the present child: (1, 0) | (2, 3); X (k1) sends g5 alone
# to the absent child: (3, 2) | (0, 1).  Unit weights: both 6/5.  w_pos = 2: X = 12/8 < Y = 12/7.  w_neg = 2: Y wins.
WBITS = np.array([[1, 1], [0, 1], [0, 1], [0, 1], [0, 1], [0, 0]])


@pytest.mark.parametrize("w_neg,w_pos,rule,T,score", [(1.0, 1.0, 0, [0, 1], 6 / 5), (1.0, 2.0, 1, [1], 12 / 8),
                                                      (2.0, 1.0, 0, [0], 12 / 8)])
def test_class_weights_change_the_split(w_neg, w_pos, rule, T, score):
    got = tree(WBITS, pos=(0, 1, 2), neg=(3, 4, 5), w_neg=w_neg, w_pos=w_pos, max_depth=1)
    assert (got[0][0], got[0][1], got[0][8]) == (rule, score, T)


def test_weighted_leaf_prediction():
    # the (1, 2) leaf predicts 1 once w_pos > 2 w_neg; at w_pos = 2, A == B and it predicts 0
    assert [n[7] for n in tree(blacklist=[1, 2], max_depth=1, w_pos=2.5)] == [1, 1, 1]
    assert [n[7] for n in tree(blacklist=[1, 2], max_depth=1, w_pos=2.0)] == [1, 1, 0]


def test_equiv_cap_truncates_but_keeps_the_total():
    assert tree(equiv_cap=1)[0][8:] == ([1], 2)
    assert tree(equiv_cap=0)[0][0] == 1 and tree(equiv_cap=0)[0][8:] == ([], 2)


def test_truncation_property_of_the_reference():
    rng = np.random.default_rng(3)
    G, U = 90, 40
    bits = (rng.random((G, U)) < 0.4).astype(np.uint8)
    labels = rng.random(G) < 0.5
    pos, neg = np.nonzero(labels)[0], np.nonzero(~labels)[0]
    m = scm_cpu.packed(bits)
    full = cart_fit(m, G, pos, neg, max_depth=None)
    assert all(n["rule"] != LEAF or n["n_pos"] == 0 or n["n_neg"] == 0 for n in full)     # distinct rows: pure leaves
    for d in (1, 2, 3):
        cut = cart_fit(m, G, pos, neg, max_depth=d)
        keep = [n for n in full if n["depth"] <= d]
        assert len(cut) == len(keep)
        for a, b in zip(cut, keep):
            assert a["n_pos"] == b["n_pos"] and a["n_neg"] == b["n_neg"]
            assert a["rule"] == (b["rule"] if b["depth"] < d else LEAF)
    # a larger min_samples_split: the same tree with the nodes of fewer examples turned into leaves
    big = cart_fit(m, G, pos, neg, max_depth=None, min_samples_split=10)
    todo = [(0, 0)]
    while todo:
        i, j = todo.pop()
        a, b = big[i], full[j]
        assert (a["n_pos"], a["n_neg"], a["depth"]) == (b["n_pos"], b["n_neg"], b["depth"])
        if a["rule"] == LEAF:
            assert b["rule"] == LEAF or a["n_pos"] + a["n_neg"] < 10
        else:
            assert a["rule"] == b["rule"]
            todo += [(a["present_child"], b["present_child"]), (a["absent_child"], b["absent_child"])]
    assert (cart_predict(full, m, G, range(G)) == labels).all()       # grown until pure on distinct rows


def test_struct_layouts_match_the_header():
    size = {"uint32_t": 4, "uint64_t": 8, "double": 8, "const uint64_t*": 8}
    for name, cls in (("grmkm_cart_job", native.CartJob), ("grmkm_cart_node", native.CartNode)):
        fields = scm_cpu._header_struct(name)
        assert [f for f, _ in cls._fields_] == [n for _, n in fields], name
        for (fname, ftype), (t, _) in zip(cls._fields_, fields):
            assert C.sizeof(ftype) == size[t], fname
        assert C.sizeof(cls) == sum(size[t] for t, _ in fields), name


def test_argument_errors_do_not_need_a_device():
    lib = native.load()
    job = native.CartJob(C.sizeof(native.CartJob), 3, 2, 0, 10, 1.0, 1.0, None, None)
    assert lib.grmkm_cart_run(None, 1, C.byref(job), None, 0) == native.E_INVALID
    assert lib.grmkm_cart_run(None, 0, None, None, 0) == native.E_INVALID
    n = C.c_uint64()
    assert lib.grmkm_cart_result(None, 0, None, 0, C.byref(n), None, 0, C.byref(n)) == native.E_INVALID


@pytest.mark.parametrize("kw", [dict(criterion="crossentropy"), dict(max_depth=0), dict(min_samples_split=1),
                                dict(class_importance={0: -1.0, 1: 1.0}), dict(class_importance={0: 1.0, 1: float("nan")}),
                                dict(class_importance={0: 1.0}), dict(max_equivalent_rules=-1)])
def test_classifier_arguments(kw):
    from grm_b200.cart import DecisionTreeClassifier
    with pytest.raises(ValueError):
        DecisionTreeClassifier(**kw)


def test_crossentropy_is_refused_with_the_reason():
    from grm_b200.cart import DecisionTreeClassifier
    with pytest.raises(ValueError, match="log"):
        DecisionTreeClassifier(criterion="crossentropy")


def test_a_multi_gpu_slice_is_refused():
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.distributed import DistributedBuilder
    from grm_b200.learning import KmerRuleClassifications
    rc = KmerRuleClassifications.__new__(KmerRuleClassifications)
    rc.builder = DistributedBuilder(n_genomes=128, rank=0, world=2, engine=object())
    with pytest.raises(ValueError, match="slice"):
        DecisionTreeClassifier().fit(rc, [0], [1])
