"""CART decision trees on the GPU-resident matrix -- Python-3 stand-in for Kover's tree learner
(bin/kover/core/kover/learning/learners/cart.py, ``kover learn tree``), gini criterion.

The reference grows a tree node by node and calls ``KmerRuleClassifications.sum_rows`` once per class for every node,
then works through all U columns with numpy on the host.  Here every level of a whole batch of trees (CV folds x class
weightings) is one pass over the resident matrix in ``grmkm_cart_run``; only the chosen splits and their equivalent
rules come back.

A node splits on a k-mer: the examples holding it go to the present child, the others to the absent child.  The score
is half the weighted Gini impurity sum of the two children, computed in a pinned order of double operations
(``include/grmkm.h``, ``DESIGN.md`` section 2), so ties and the chosen k-mer (the lowest column index of the tie set)
do not depend on the GPU, the batch or the grid.

The tree fitted with ``max_depth = d`` is the depth-d truncation of the tree fitted with any larger ``max_depth``, and
a larger ``min_samples_split`` only turns internal nodes into leaves, so a max-depth or min-samples grid needs one tree
per fold and class weighting; ``model_selection.cross_validate_cart`` scores such a grid from one tree per fold and
picks its hyperparameters.  Cost-complexity pruning is the caller's.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np

from .scm import KmerRule, _kmer_string, _refuse_slices

# rule: the split's KmerRule (type "presence": its examples go to present_child), None for a leaf.  prediction: the
# leaf's output (1 iff w_pos * n_pos > w_neg * n_neg).  equivalent_rules: the k-mer indices of the splits tied with it
# (at most max_equivalent_rules, the smallest), equivalent_total: how many tie in all.
Node = namedtuple("Node", "rule score depth n_pos n_neg present_child absent_child prediction equivalent_rules "
                          "equivalent_total")

_UNLIMITED_DEPTH = 2**32 - 1
_ALL_EQUIVALENT = 2**64 - 1
_MAX_IMPORTANCE = 1e100         # larger class importances could overflow the products of the score


class DecisionTreeClassifier:
    def __init__(self, criterion: str = "gini", max_depth: int | None = 10, min_samples_split: int = 2,
                 class_importance: dict | None = None, max_equivalent_rules: int | None = None):
        if criterion != "gini":
            raise ValueError(f"criterion must be 'gini', not {criterion!r}: an entropy score needs log, whose last bit "
                             "differs between the GPU and the host library, so its ties could not be reproduced exactly")
        if max_depth is not None and int(max_depth) < 1:
            raise ValueError("max_depth must be at least 1 (or None: grow until the leaves are pure)")
        if int(min_samples_split) < 2:
            raise ValueError("min_samples_split must be at least 2")
        ci = {0: 1.0, 1: 1.0} if class_importance is None else dict(class_importance)
        if set(ci) != {0, 1}:
            raise ValueError("class_importance maps the classes 0 and 1 to their weights")
        ci = {k: float(v) for k, v in ci.items()}
        if not all(np.isfinite(v) and 0 < v <= _MAX_IMPORTANCE for v in ci.values()):
            raise ValueError(f"class importances must be finite, > 0 and <= {_MAX_IMPORTANCE:g}, not {ci}")
        if max_equivalent_rules is not None and int(max_equivalent_rules) < 0:
            raise ValueError("max_equivalent_rules must be >= 0 (or None: all of them)")
        self.criterion = criterion
        self.max_depth = None if max_depth is None else int(max_depth)
        self.min_samples_split = int(min_samples_split)
        self.class_importance = ci
        self.max_equivalent_rules = None if max_equivalent_rules is None else int(max_equivalent_rules)
        self.nodes: list[Node] = []              # breadth-first: the root is 0, children follow their parents' order

    def fit(self, rule_classifications, positive_example_idx, negative_example_idx, rule_blacklist=None):
        """Learn from the examples (row indices among the rows not removed, as in sum_rows).  rule_blacklist: rule
        indices; j or U + j removes k-mer j from the candidate splits."""
        fit_many(rule_classifications, [(self, positive_example_idx, negative_example_idx)], rule_blacklist)
        return self

    def predict(self, rule_classifications, example_idx) -> np.ndarray:
        """0/1 per example (row indices among the rows not removed): the examples walk the tree from the root, on the
        columns of the tree's split k-mers only."""
        if not self.nodes:
            raise ValueError("the tree is not fitted")
        example_idx = np.asarray(example_idx, dtype=np.int64).reshape(-1)
        kmers = sorted({x.rule.kmer_index for x in self.nodes if x.rule is not None})
        col_of = {j: i for i, j in enumerate(kmers)}
        col = np.array([col_of[x.rule.kmer_index] if x.rule is not None else -1 for x in self.nodes], dtype=np.int64)
        cols = (rule_classifications.get_columns(kmers)[example_idx] if kmers
                else np.zeros((len(example_idx), 0), dtype=np.uint8))
        return _tree_output(self.nodes, col, cols)

    def predict_genomes(self, builder) -> np.ndarray:
        """0/1 per genome row of the inputs of ``builder`` (a KmerMatrixBuilder holding genomes that need not have
        been in the training matrix): one ``builder.query`` of the split k-mers, no build (predict.predict_genomes)."""
        from .predict import predict_genomes
        return predict_genomes([self], builder)[0]


def _tree_output(nodes, col: np.ndarray, cols: np.ndarray) -> np.ndarray:
    """The leaf prediction of every example: cols = 0/1 (examples x columns), col[i] = the column of node i's split
    k-mer (-1: a leaf).  The examples walk the tree from the root to their leaves."""
    n = len(nodes)
    present = np.array([-1 if x.rule is None else x.present_child for x in nodes], dtype=np.int64)
    absent = np.array([-1 if x.rule is None else x.absent_child for x in nodes], dtype=np.int64)
    pred = np.array([x.prediction for x in nodes], dtype=np.uint8)
    at = np.zeros(len(cols), dtype=np.int64)
    for _ in range(n):
        inner = np.nonzero(col[at] >= 0)[0]
        if not len(inner):
            break
        here = at[inner]
        at[inner] = np.where(cols[inner, col[here]] == 1, present[here], absent[here])
    return pred[at]


def fit_many(rule_classifications, trees, rule_blacklist=None):
    """Grow every (tree, positive_example_idx, negative_example_idx) of ``trees`` to completion in one batch on the GPU
    (one pass over the matrix per level of all pending trees).  The trees get their nodes."""
    _refuse_slices(rule_classifications)
    rc = rule_classifications
    b = rc.builder
    jobs = []
    for t, pos, neg in trees:
        jobs.append((_UNLIMITED_DEPTH if t.max_depth is None else t.max_depth, t.min_samples_split,
                     _ALL_EQUIVALENT if t.max_equivalent_rules is None else t.max_equivalent_rules,
                     t.class_importance[0], t.class_importance[1], rc.row_mask(pos), rc.row_mask(neg)))
    blacklist = np.asarray(rule_blacklist if rule_blacklist is not None else [], dtype=np.uint64).reshape(-1)
    results = b.cart_run(jobs, blacklist, shard=rc.shard)
    needed = sorted({int(x["rule"]) for nodes, _ in results for x in nodes if int(x["present_child"]) != 0xFFFFFFFF})
    seqs = dict(zip(needed, (_kmer_string(int(x), b.k) for x in rc.kmers_at(needed)))) if needed else {}
    for (t, _, _), (nodes, eq) in zip(trees, results):
        t.nodes = []
        for x in nodes:
            rule = None
            if int(x["present_child"]) != 0xFFFFFFFF:
                j = int(x["rule"])
                rule = KmerRule(j, seqs[j], "presence")
            o, c = int(x["equiv_offset"]), int(x["equiv_count"])
            t.nodes.append(Node(rule, float(x["score"]), int(x["depth"]), int(x["n_pos"]), int(x["n_neg"]),
                                _child(x["present_child"]), _child(x["absent_child"]), int(x["prediction"]),
                                eq[o:o + c].astype(np.int64), int(x["equiv_total"])))
    return [t for t, _, _ in trees]


def _child(v) -> int | None:
    v = int(v)
    return None if v == 0xFFFFFFFF else v
