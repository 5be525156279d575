"""CPU: the host side of cross-validated selection (grm_b200.model_selection) -- folds, the count tables, the selection
rules, metrics and tree truncation on hand-built inputs -- and the numpy reference of grmkm_eval_run on hand cases."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from grm_b200 import model_selection as ms
from grm_b200 import native
from grm_b200.cart import DecisionTreeClassifier, Node
from grm_b200.scm import KmerRule
from tests.eval_oracle import LEAF, eval_cart, eval_scm


# -- folds ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n_pos,n_neg,k", [(7, 13, 5), (5, 5, 2), (10, 1, 3), (3, 0, 3), (100, 37, 10)])
def test_folds_are_stratified_and_balanced(n_pos, n_neg, k):
    labels = np.array([1] * n_pos + [0] * n_neg)
    f = ms.make_folds(labels, k, 3)
    assert f.shape == labels.shape and set(f.tolist()) <= set(range(k))
    for c in (0, 1):
        sizes = np.bincount(f[labels == c], minlength=k)
        assert sizes.max() - sizes.min() <= 1
    sizes = np.bincount(f, minlength=k)
    assert sizes.min() >= 1 and sizes.max() - sizes.min() <= 1


def test_folds_are_deterministic_per_seed():
    labels = np.array([1, 0] * 50)
    assert np.array_equal(ms.make_folds(labels, 5, 7), ms.make_folds(labels, 5, 7))
    assert not np.array_equal(ms.make_folds(labels, 5, 7), ms.make_folds(labels, 5, 8))


def test_fold_arguments_are_validated():
    labels = np.array([1, 1, 0, 0])
    with pytest.raises(ValueError):
        ms.make_folds(labels, 1, 0)
    with pytest.raises(ValueError):
        ms.make_folds(labels, 5, 0)                          # a fold would be empty
    ids, k = ms._fold_ids([0, 1, 1, 0], labels, 0)
    assert k == 2 and ids.tolist() == [0, 1, 1, 0]
    for bad in ([0, 0, 0, 0], [0, 2, 2, 0], [0, 1, 1], [0, 1, -1, 0], [0.0, 1.0, 1.0, 0.0]):
        with pytest.raises(ValueError):
            ms._fold_ids(bad, labels, 0)
    ids, k = ms._fold_ids(2, labels, 0)
    assert k == 2 and np.array_equal(ids, ms.make_folds(labels, 2, 0))


# -- SCM tables and selection -----------------------------------------------------------------------------------------

def test_scm_cv_errors_score_a_short_fit_at_its_last_prefix():
    # 2 folds x 2 candidates; candidate 1 of fold 0 stopped after 1 rule
    f0 = [np.array([[5, 0], [2, 1], [1, 1], [0, 1]]), np.array([[0, 9], [3, 0]])]
    f1 = [np.array([[4, 0], [1, 2], [1, 0], [0, 0]]), np.array([[0, 8], [2, 2], [2, 1], [2, 1]])]
    err = ms._scm_cv_errors([f0, f1], 3)
    assert err.tolist() == [[3 + 3, 2 + 1, 1 + 0], [3 + 4, 3 + 3, 3 + 3]]
    assert err.dtype == np.int64


def test_scm_selection_tie_breaks():
    e = np.full((2, 3, 4), 9, dtype=np.int64)              # (type, p, r - 1)
    e[1, 2, 3] = 2
    assert ms._select_scm(e) == (1, 2, 4)                  # least error wins
    e[1, 1, 3] = 2
    assert ms._select_scm(e) == (1, 1, 4)                  # tie: earlier p
    e[0, 2, 3] = 2
    assert ms._select_scm(e) == (0, 2, 4)                  # tie: earlier model type before earlier p
    e[1, 2, 1] = 2
    assert ms._select_scm(e) == (1, 2, 2)                  # tie: fewer rules first
    e[:] = 0
    assert ms._select_scm(e) == (0, 0, 1)


# -- metrics --------------------------------------------------------------------------------------------------------

def test_metrics():
    m = ms.confusion_metrics(10, 20, 2, 5)
    assert (m["tp"], m["fn"], m["fp"], m["tn"]) == (8, 2, 5, 15)
    assert m["risk"] == 7 / 30 and m["sensitivity"] == 8 / 10 == m["recall"] and m["specificity"] == 15 / 20
    assert m["precision"] == 8 / 13 and m["f1"] == 16 / 23


def test_metrics_zero_denominators():
    m = ms.confusion_metrics(0, 0, 0, 0)
    assert all(m[k] is None for k in ("risk", "sensitivity", "specificity", "precision", "recall", "f1"))
    m = ms.confusion_metrics(0, 4, 0, 0)                    # no positives, none called positive
    assert m["risk"] == 0 and m["specificity"] == 1 and m["sensitivity"] is None and m["precision"] is None
    assert m["f1"] is None
    m = ms.confusion_metrics(3, 0, 3, 0)                    # every positive missed
    assert m["sensitivity"] == 0 and m["precision"] is None and m["f1"] == 0 and m["specificity"] is None


# -- trees ----------------------------------------------------------------------------------------------------------

def _node(rule, depth, a, b, pc=None, ac=None, pred=None):
    r = None if rule is None else KmerRule(rule, "A" * 3, "presence")
    return Node(r, 0.0 if rule is None else 0.25, depth, a, b, pc, ac, int(a > b) if pred is None else pred,
                np.array([] if rule is None else [rule], dtype=np.int64), 0 if rule is None else 1)


# a grown tree: 0 -> (1, 2), 1 -> (3, 4), 2 leaf, 3 -> (5, 6), 4 leaf, 5 leaf, 6 leaf
TREE = [_node(7, 0, 6, 6, 1, 2), _node(3, 1, 5, 2, 3, 4), _node(None, 1, 1, 4), _node(9, 2, 2, 2, 5, 6),
        _node(None, 2, 3, 0), _node(None, 3, 2, 0), _node(None, 3, 0, 2)]


@pytest.mark.parametrize("d,s,kept,leaves", [
    (None, 2, [0, 1, 2, 3, 4, 5, 6], [2, 4, 5, 6]),
    (3, 2, [0, 1, 2, 3, 4, 5, 6], [2, 4, 5, 6]),
    (2, 2, [0, 1, 2, 3, 4], [2, 3, 4]),
    (1, 2, [0, 1, 2], [1, 2]),
    (None, 5, [0, 1, 2, 3, 4], [2, 3, 4]),                 # node 3 holds 4 training examples < 5
    (None, 8, [0, 1, 2], [1, 2]),                          # node 1 holds 7 < 8
    (None, 13, [0], [0]),
])
def test_truncation_leaves(d, s, kept, leaves):
    k, leaf = ms._truncation(ms._node_table(TREE), d, s)
    assert np.nonzero(k)[0].tolist() == kept and np.nonzero(leaf)[0].tolist() == leaves


def test_tree_errors_from_node_counts():
    counts = np.array([[9, 8], [6, 3], [3, 5], [4, 1], [2, 2], [3, 0], [1, 1]])
    table = ms._node_table(TREE)
    # predictions (a > b) of nodes 0..6: 0, 1, 0, 0, 1, 1, 0; fn = pos at leaves predicting 0, fp = neg at leaves predicting 1
    assert ms._tree_errors(table, counts, None, 2) == (3 + 1, 2 + 0)
    assert ms._tree_errors(table, counts, 2, 2) == (3 + 4, 2)           # leaves 2 (pred 0), 3 (pred 0), 4 (pred 1)
    assert ms._tree_errors(table, counts, 1, 2) == (3, 3)               # leaves 1 (pred 1), 2 (pred 0)
    assert ms._tree_errors(table, counts, None, 13) == (9, 0)           # the root alone: 6 vs 6 predicts 0


def test_truncated_tree_is_renumbered_breadth_first():
    t = DecisionTreeClassifier(max_depth=None)
    t.nodes = list(TREE)
    out = ms._truncate(t, 2, 2)
    assert out.max_depth == 2 and out.min_samples_split == 2 and len(out.nodes) == 5
    assert out.nodes[3].rule is None and out.nodes[3].present_child is None and out.nodes[3].score == 0.0
    assert out.nodes[3].equivalent_total == 0 and len(out.nodes[3].equivalent_rules) == 0
    assert [(x.present_child, x.absent_child) for x in out.nodes[:2]] == [(1, 2), (3, 4)]
    # a deeper cut keeps node 3's children, renumbered 5 and 6
    t2 = ms._truncate(t, None, 3)
    assert [x.present_child for x in t2.nodes] == [1, 3, None, 5, None, None, None]
    # drop node 1's subtree: node 2's index stays, node 1 becomes a leaf
    t3 = ms._truncate(t, None, 8)
    assert len(t3.nodes) == 3 and t3.nodes[1].rule is None and t3.nodes[0].absent_child == 2


def test_cart_selection_tie_breaks():
    depths, mss = [3, None, 1], [2, 10, 5]
    e = np.full((2, 3, 3), 9, dtype=np.int64)              # (weighting, depth, min samples)
    e[1, 1, 0] = 4
    assert ms._select_cart(e, depths, mss) == (1, 1, 0)
    e[1, 0, 0] = 4
    assert ms._select_cart(e, depths, mss) == (1, 0, 0)    # depth 3 before unlimited
    e[1, 2, 0] = 4
    assert ms._select_cart(e, depths, mss) == (1, 2, 0)    # depth 1 first
    e[1, 2, 2] = 4
    assert ms._select_cart(e, depths, mss) == (1, 2, 2)    # larger min_samples_split (5 > 2)
    e[0, 2, 0] = 4
    assert ms._select_cart(e, depths, mss) == (1, 2, 2)    # depth and min samples come before the weighting
    e[0, 2, 2] = 4
    assert ms._select_cart(e, depths, mss) == (0, 2, 2)
    e[1, 2, 1] = 3
    assert ms._select_cart(e, depths, mss) == (1, 2, 1)


# -- the numpy reference of grmkm_eval_run ----------------------------------------------------------------------------

BITS = np.array([[1, 0, 1],
                 [1, 1, 0],
                 [0, 1, 1],
                 [0, 0, 0],
                 [1, 1, 1]], dtype=np.uint8)               # 5 genomes x 3 k-mers; rule 3 + j = "k-mer j absent"


def test_reference_scm_prefixes():
    pos, neg = [0, 1, 4], [2, 3]
    # conjunction of k-mer 0 present, then k-mer 2 absent: outputs 11111 -> 11001 -> 01000
    assert eval_scm(BITS, "conjunction", [0, 5], pos, neg).tolist() == [[0, 2], [0, 0], [2, 0]]
    # disjunction of k-mer 1 present, then k-mer 0 absent: 00000 -> 01101 -> 01111
    assert eval_scm(BITS, "disjunction", [1, 3], pos, neg).tolist() == [[3, 0], [1, 1], [1, 2]]
    assert eval_scm(BITS, "conjunction", [], pos, neg).tolist() == [[0, 2]]
    assert eval_scm(BITS, "disjunction", [], [], []).tolist() == [[0, 0]]


def test_reference_tree_counts():
    # root splits on k-mer 0: present -> node 1 (split on k-mer 2), absent -> node 2 (leaf); node 1 -> 3, 4
    nodes = [(0, 1, 2), (2, 3, 4), (LEAF, 0, 0), (LEAF, 0, 0), (LEAF, 0, 0)]
    got = eval_cart(BITS, nodes, [0, 1, 4], [2, 3])
    assert got.tolist() == [[3, 2], [3, 0], [0, 2], [2, 0], [1, 0]]
    assert eval_cart(BITS, [(LEAF, 0, 0)], [0], [1, 2]).tolist() == [[1, 2]]


def test_eval_structs_match_the_header():
    assert C.sizeof(native.EvalNode) == 16
    assert C.sizeof(native.EvalJob) == 4 * 4 + 8 + 4 * 8
    from grm_b200.builder import KmerMatrixBuilder
    assert KmerMatrixBuilder.EVAL_NODE_DTYPE.itemsize == C.sizeof(native.EvalNode)


def test_slices_are_refused():
    rc = SimpleNamespace(builder=SimpleNamespace(world=2))
    with pytest.raises(ValueError, match="slice"):
        ms.cross_validate_scm(rc, [0], [1], ["conjunction"], [1.0], 2, 2)
    with pytest.raises(ValueError, match="slice"):
        ms.cross_validate_cart(rc, [0], [1], [None], [1], [2], 2)
