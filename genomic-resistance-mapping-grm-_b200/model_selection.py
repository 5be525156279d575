"""Hyperparameter selection by cross-validation for the Set Covering Machine and CART on the GPU-resident matrix --
the ``--hp-choice cv`` path of ``kover learn scm|tree``: fit the grid on the CV folds, score every candidate on the
held-out examples, pick one, take the model of the whole training set, report train / test metrics.

Per learner one batched fit (``scm.fit_many`` / ``cart.fit_many``: every fold's training part and the whole training
set) and one ``KmerMatrixBuilder.eval_run`` (``grmkm_eval_run``) that scores all folds' models on their held-out
examples, and the whole-set models on the training and test sets, in one launch.  Only counts come back: the matrix
never leaves the GPU and no column is unpacked on the host.

Examples are row indices among the rows not removed, as in ``sum_rows``.  The training examples are numbered
``train_pos`` first, then ``train_neg``; explicit fold ids (``folds`` as an array) follow that order.  Folds and the
selection rules are restated here (DESIGN.md section 2), not Kover's random stream: the same seed gives the same folds
here, not the folds Kover would draw.
"""
from __future__ import annotations

import time

import numpy as np

from . import cart, native, scm
from .scm import SetCoveringMachine, _refuse_slices


def make_folds(labels, n_folds: int, random_seed: int = 0) -> np.ndarray:
    """Stratified fold ids (0..n_folds-1), one per example of ``labels``: the examples of each class (ascending class
    order) are permuted by ``np.random.default_rng(random_seed)`` and dealt to the folds round-robin, the dealing of a
    class continuing where the previous class stopped.  So per class, and overall, fold sizes differ by at most one."""
    labels = np.asarray(labels).reshape(-1)
    n_folds = int(n_folds)
    if n_folds < 2:
        raise ValueError("n_folds must be at least 2")
    if n_folds > len(labels):
        raise ValueError(f"{n_folds} folds for {len(labels)} examples: a fold would be empty")
    rng = np.random.default_rng(random_seed)
    fold = np.empty(len(labels), dtype=np.int64)
    start = 0
    for c in np.unique(labels):
        idx = rng.permutation(np.nonzero(labels == c)[0])
        fold[idx] = (start + np.arange(len(idx))) % n_folds
        start += len(idx)
    return fold


def _fold_ids(folds, labels, random_seed) -> tuple[np.ndarray, int]:
    """(fold id per training example, number of folds) from a fold count or explicit ids."""
    if np.ndim(folds) == 0:
        ids = make_folds(labels, int(folds), random_seed)
        return ids, int(folds)
    ids = np.asarray(folds)
    if ids.shape != (len(labels),):
        raise ValueError(f"{ids.size} fold ids for {len(labels)} training examples")
    if len(ids) and not np.issubdtype(ids.dtype, np.integer):
        raise ValueError("fold ids must be integers")
    ids = ids.astype(np.int64)
    k = int(ids.max()) + 1 if len(ids) else 0
    if k < 2 or ids.min() < 0 or len(np.unique(ids)) != k:
        raise ValueError("fold ids must be 0..k-1 with k >= 2 and no fold empty")
    return ids, k


def confusion_metrics(n_pos: int, n_neg: int, fn: int, fp: int) -> dict:
    """Confusion counts and metrics of a model on n_pos positive and n_neg negative examples, of which it misses fn
    positives and calls fp negatives positive.  Each rate is None when its denominator is 0."""
    n_pos, n_neg, fn, fp = int(n_pos), int(n_neg), int(fn), int(fp)
    tp, tn = n_pos - fn, n_neg - fp

    def ratio(a, b):
        return a / b if b else None

    return {"n_pos": n_pos, "n_neg": n_neg, "tp": tp, "fn": fn, "fp": fp, "tn": tn,
            "risk": ratio(fn + fp, n_pos + n_neg), "sensitivity": ratio(tp, tp + fn), "specificity": ratio(tn, tn + fp),
            "precision": ratio(tp, tp + fp), "recall": ratio(tp, tp + fn), "f1": ratio(2 * tp, 2 * tp + fp + fn)}


class SelectionResult:
    """What a cross-validated selection found.  ``grid``: one dict per candidate (its hyperparameters, ``cv_errors``
    -- the integer sum over the folds of the held-out errors -- and ``cv_risk`` = cv_errors / training examples);
    ``selected``: the chosen candidate's dict; ``model``: the whole-training-set model with those hyperparameters;
    ``train`` / ``test``: confusion_metrics of the model (test: None without a test set); ``seconds``: wall time of
    the batched fit, of the evaluation pass and of the whole call."""

    def __init__(self, learner, n_folds, fold_ids, grid, selected, model, train, test, seconds):
        self.learner, self.n_folds, self.fold_ids = learner, n_folds, fold_ids
        self.grid, self.selected, self.model = grid, selected, model
        self.train, self.test, self.seconds = train, test, seconds

    def to_dict(self) -> dict:
        """JSON-serialisable form (the model as its rules or nodes)."""
        return {"learner": self.learner, "n_folds": self.n_folds, "fold_ids": [int(x) for x in self.fold_ids],
                "grid": self.grid, "selected": self.selected, "model": _model_dict(self.model), "train": self.train,
                "test": self.test, "seconds": self.seconds}


def _model_dict(m) -> dict:
    if isinstance(m, SetCoveringMachine):
        return {"model_type": m.model_type, "p": m.p, "max_rules": m.max_rules,
                "rule_indices": [int(r) for r in m.rule_indices],
                "rules": [{"kmer_index": int(r.kmer_index), "kmer_sequence": r.kmer_sequence, "type": r.type}
                          for r in m.model]}
    return {"max_depth": m.max_depth, "min_samples_split": m.min_samples_split,
            "class_importance": {str(k): v for k, v in m.class_importance.items()},
            "nodes": [{"kmer_index": None if x.rule is None else int(x.rule.kmer_index),
                       "kmer_sequence": None if x.rule is None else x.rule.kmer_sequence, "score": x.score,
                       "depth": x.depth, "n_pos": x.n_pos, "n_neg": x.n_neg, "present_child": x.present_child,
                       "absent_child": x.absent_child, "prediction": x.prediction,
                       "equivalent_rules": [int(r) for r in x.equivalent_rules], "equivalent_total": x.equivalent_total}
                      for x in m.nodes]}


def _split(rc, train_pos, train_neg, folds, random_seed):
    pos = np.asarray(train_pos, dtype=np.int64).reshape(-1)
    neg = np.asarray(train_neg, dtype=np.int64).reshape(-1)
    labels = np.concatenate([np.ones(len(pos), dtype=np.int64), np.zeros(len(neg), dtype=np.int64)])
    ids, k = _fold_ids(folds, labels, random_seed)
    # set s < k: fold s's training part and its held-out part; set k: the whole training set
    sets = [(pos[ids[:len(pos)] != f], neg[ids[len(pos):] != f], pos[ids[:len(pos)] == f], neg[ids[len(pos):] == f])
            for f in range(k)]
    sets.append((pos, neg, pos, neg))
    return pos, neg, ids, k, sets


# -- Set Covering Machine -----------------------------------------------------------------------------------------

def _scm_cv_errors(fold_counts, max_rules: int) -> np.ndarray:
    """fold_counts[f][c]: (R_fc + 1, 2) held-out (fn, fp) of candidate machine c of fold f by prefix length.  ->
    errors[c, r - 1] for r = 1..max_rules: the sum over folds of fn + fp at prefix min(r, R_fc) (int64)."""
    n_cand = len(fold_counts[0]) if fold_counts else 0
    err = np.zeros((n_cand, max_rules), dtype=np.int64)
    r = np.arange(1, max_rules + 1)
    for per_fold in fold_counts:
        for c, cnt in enumerate(per_fold):
            tot = np.asarray(cnt, dtype=np.int64).sum(axis=1)
            err[c] += tot[np.minimum(r, len(tot) - 1)]
    return err


def _select_scm(errors: np.ndarray) -> tuple[int, int, int]:
    """errors[t, p, r - 1] (integers) -> (t, p, r) of least error; ties: fewest rules, then t, then p (their order)."""
    best = errors.min()
    t, p, r = np.nonzero(errors == best)
    i = np.lexsort((p, t, r))[0]
    return int(t[i]), int(p[i]), int(r[i]) + 1


def _cut(m: SetCoveringMachine, r: int) -> SetCoveringMachine:
    """The machine's first r rules as a machine of max_rules = r (the greedy steps do not depend on max_rules)."""
    out = SetCoveringMachine(m.model_type, m.p, r)
    out.model, out.iterations, out.rule_indices = m.model[:r], m.iterations[:r], m.rule_indices[:r]
    return out


def cross_validate_scm(rc, train_pos, train_neg, model_types, p_values, max_rules, folds, random_seed=0,
                       rule_blacklist=None, test_pos=(), test_neg=()) -> SelectionResult:
    """Choose (model type, p, number of rules) by k-fold CV and return the whole-training-set machine with them.

    folds: the number of stratified folds (make_folds with random_seed) or one fold id per training example.  One
    fit_many fits (k + 1) x |model_types| x |p_values| machines with max_rules rules; one eval_run scores every fold's
    machines on that fold's held-out examples at every prefix, and the whole-set machines on the training and test
    sets.  A fold's machine that stopped after R_f < r rules is scored at R_f.  Least integer CV error wins; ties go to
    fewer rules, then the order of model_types, then the order of p_values."""
    _refuse_slices(rc)
    t_start = time.perf_counter()
    model_types, p_values, max_rules = list(model_types), [float(p) for p in p_values], int(max_rules)
    if not model_types or not p_values:
        raise ValueError("model_types and p_values must not be empty")
    pos, neg, ids, k, sets = _split(rc, train_pos, train_neg, folds, random_seed)
    test_pos = np.asarray(test_pos, dtype=np.int64).reshape(-1)
    test_neg = np.asarray(test_neg, dtype=np.int64).reshape(-1)
    has_test = len(test_pos) + len(test_neg) > 0
    nT, nP = len(model_types), len(p_values)
    machines = [[SetCoveringMachine(t, p, max_rules) for t in model_types for p in p_values] for _ in sets]

    t0 = time.perf_counter()
    scm.fit_many(rc, [(m, s[0], s[1]) for ms, s in zip(machines, sets) for m in ms], rule_blacklist)
    t_fit = time.perf_counter() - t0

    eval_sets = [(s[2], s[3]) for s in sets]
    if has_test:
        eval_sets.append((test_pos, test_neg))
    masks = [(rc.row_mask(a), rc.row_mask(b)) for a, b in eval_sets]
    jobs = []
    for e, (pm, nm) in enumerate(masks):
        for m in machines[min(e, k)]:
            jobs.append((native.EVAL_SCM, scm._MODEL_TYPES[m.model_type], m.rule_indices, pm, nm))
    t0 = time.perf_counter()
    counts = rc.builder.eval_run(jobs, shard=rc.shard)
    t_eval = time.perf_counter() - t0

    n_cand = nT * nP
    per_set = [counts[e * n_cand:(e + 1) * n_cand] for e in range(len(masks))]
    errors = _scm_cv_errors(per_set[:k], max_rules).reshape(nT, nP, max_rules)
    m_train = len(pos) + len(neg)
    grid = [{"model_type": model_types[t], "p": p_values[p], "max_rules": r + 1, "cv_errors": int(errors[t, p, r]),
             "cv_risk": errors[t, p, r] / m_train if m_train else None}
            for r in range(max_rules) for t in range(nT) for p in range(nP)]
    t, p, r = _select_scm(errors)
    selected = next(g for g in grid if g["model_type"] == model_types[t] and g["p"] == p_values[p] and g["max_rules"] == r)
    full = machines[k][t * nP + p]
    model = _cut(full, min(r, len(full.rule_indices)))
    rr = len(model.rule_indices)

    def metrics(e, a, b):
        fn, fp = per_set[e][t * nP + p][rr]
        return confusion_metrics(len(a), len(b), fn, fp)

    return SelectionResult("scm", k, ids, grid, selected, model, metrics(k, pos, neg),
                           metrics(k + 1, test_pos, test_neg) if has_test else None,
                           {"fit": t_fit, "eval": t_eval, "total": time.perf_counter() - t_start})


# -- CART -----------------------------------------------------------------------------------------------------------

def _node_table(nodes):
    """Arrays of a fitted tree's nodes: split (bool), depth, training examples, present / absent child, prediction."""
    split = np.array([x.rule is not None for x in nodes], dtype=bool)
    depth = np.array([x.depth for x in nodes], dtype=np.int64)
    n = np.array([x.n_pos + x.n_neg for x in nodes], dtype=np.int64)
    present = np.array([x.present_child if x.rule is not None else -1 for x in nodes], dtype=np.int64)
    absent = np.array([x.absent_child if x.rule is not None else -1 for x in nodes], dtype=np.int64)
    pred = np.array([x.prediction for x in nodes], dtype=np.int64)
    return split, depth, n, present, absent, pred


def _truncation(table, max_depth, min_samples_split) -> tuple[np.ndarray, np.ndarray]:
    """(kept, leaf) masks of the (max_depth, min_samples_split) truncation of a tree (max_depth None: no limit): a
    reached node is a leaf if it is a leaf of the tree, sits at depth max_depth, or holds fewer than min_samples_split
    training examples; the children of a leaf are not reached."""
    split, depth, n, present, absent, _ = table
    kept = np.zeros(len(split), dtype=bool)
    leaf = np.zeros(len(split), dtype=bool)
    if not len(split):
        return kept, leaf
    kept[0] = True
    for i in range(len(split)):          # a child's index is above its parent's: one pass in index order
        if not kept[i]:
            continue
        if not split[i] or (max_depth is not None and depth[i] >= max_depth) or n[i] < min_samples_split:
            leaf[i] = True
        else:
            kept[present[i]] = kept[absent[i]] = True
    return kept, leaf


def _tree_errors(table, counts, max_depth, min_samples_split) -> tuple[int, int]:
    """(fn, fp) of the truncation from per-node counts (pos, neg reaching each node of the grown tree)."""
    _, leaf = _truncation(table, max_depth, min_samples_split)
    pred = table[5]
    counts = np.asarray(counts, dtype=np.int64)
    return int(counts[leaf & (pred == 0), 0].sum()), int(counts[leaf & (pred == 1), 1].sum())


def _select_cart(errors: np.ndarray, max_depths, min_samples_splits) -> tuple[int, int, int]:
    """errors[w, d, s] (integers) -> (w, d, s) of least error; ties: smaller depth (None is the largest), then larger
    min_samples_split, then w (the order of the weightings), then the order the values were given in."""
    best = errors.min()
    w, d, s = np.nonzero(errors == best)
    depth_key = np.array([np.inf if max_depths[i] is None else max_depths[i] for i in d], dtype=np.float64)
    mss_key = -np.array([min_samples_splits[i] for i in s], dtype=np.float64)
    i = np.lexsort((s, d, w, mss_key, depth_key))[0]
    return int(w[i]), int(d[i]), int(s[i])


def _truncate(tree, max_depth, min_samples_split):
    """The truncated tree as a DecisionTreeClassifier of those hyperparameters, its nodes renumbered breadth-first;
    a node that became a leaf has no rule, score 0, no equivalent rules and no children."""
    kept, leaf = _truncation(_node_table(tree.nodes), max_depth, min_samples_split)
    new_index = np.cumsum(kept) - 1          # kept nodes keep their breadth-first order
    out = cart.DecisionTreeClassifier(tree.criterion, max_depth, min_samples_split, tree.class_importance,
                                      tree.max_equivalent_rules)
    for i in np.nonzero(kept)[0]:
        x = tree.nodes[i]
        if leaf[i]:
            x = x._replace(rule=None, score=0.0, present_child=None, absent_child=None,
                           equivalent_rules=np.zeros(0, dtype=np.int64), equivalent_total=0)
        else:
            x = x._replace(present_child=int(new_index[x.present_child]), absent_child=int(new_index[x.absent_child]))
        out.nodes.append(x)
    return out


def _eval_nodes(nodes) -> np.ndarray:
    from .builder import KmerMatrixBuilder
    arr = np.zeros(len(nodes), dtype=KmerMatrixBuilder.EVAL_NODE_DTYPE)
    for i, x in enumerate(nodes):
        if x.rule is None:
            arr[i] = (np.iinfo(np.uint64).max, 0xFFFFFFFF, 0xFFFFFFFF)
        else:
            arr[i] = (x.rule.kmer_index, x.present_child, x.absent_child)
    return arr


def cross_validate_cart(rc, train_pos, train_neg, class_importances, max_depths, min_samples_splits, folds,
                        random_seed=0, rule_blacklist=None, max_equivalent_rules=None, test_pos=(),
                        test_neg=()) -> SelectionResult:
    """Choose (class importance, max_depth, min_samples_split) by k-fold CV and return the truncated
    whole-training-set tree.

    class_importances: dicts {0: w_neg, 1: w_pos} (None: unit weights); max_depths: ints >= 1 or None (no limit).
    folds as in cross_validate_scm.  One fit_many grows a tree per (fold set, weighting) with the largest max_depth and
    the smallest min_samples_split; the (depth, min-samples) grid is scored from per-node held-out counts of one
    eval_run, since the tree of (d, s) is the truncation of the grown tree (DESIGN.md section 2).  Least integer CV
    error wins; ties go to the smaller depth, then the larger min_samples_split, then the order of the weightings."""
    _refuse_slices(rc)
    t_start = time.perf_counter()
    weights = [None if ci is None else dict(ci) for ci in class_importances]
    max_depths = [None if d is None else int(d) for d in max_depths]
    mss = [int(s) for s in min_samples_splits]
    if not weights or not max_depths or not mss:
        raise ValueError("class_importances, max_depths and min_samples_splits must not be empty")
    grow_depth = None if any(d is None for d in max_depths) else max(max_depths)
    pos, neg, ids, k, sets = _split(rc, train_pos, train_neg, folds, random_seed)
    for d in max_depths:                 # the classifier checks the values it is given; check every grid value
        cart.DecisionTreeClassifier(max_depth=d)
    for s in mss:
        cart.DecisionTreeClassifier(min_samples_split=s)
    test_pos = np.asarray(test_pos, dtype=np.int64).reshape(-1)
    test_neg = np.asarray(test_neg, dtype=np.int64).reshape(-1)
    has_test = len(test_pos) + len(test_neg) > 0
    trees = [[cart.DecisionTreeClassifier("gini", grow_depth, min(mss), ci, max_equivalent_rules) for ci in weights]
             for _ in sets]

    t0 = time.perf_counter()
    cart.fit_many(rc, [(t, s[0], s[1]) for ts, s in zip(trees, sets) for t in ts], rule_blacklist)
    t_fit = time.perf_counter() - t0

    eval_sets = [(s[2], s[3]) for s in sets]
    if has_test:
        eval_sets.append((test_pos, test_neg))
    jobs = []
    for e, (a, b) in enumerate(eval_sets):
        pm, nm = rc.row_mask(a), rc.row_mask(b)
        for t in trees[min(e, k)]:
            jobs.append((native.EVAL_CART, 0, _eval_nodes(t.nodes), pm, nm))
    t0 = time.perf_counter()
    counts = rc.builder.eval_run(jobs, shard=rc.shard)
    t_eval = time.perf_counter() - t0

    nW = len(weights)
    per_set = [counts[e * nW:(e + 1) * nW] for e in range(len(eval_sets))]
    errors = np.zeros((nW, len(max_depths), len(mss)), dtype=np.int64)
    for f in range(k):
        for w in range(nW):
            table = _node_table(trees[f][w].nodes)
            for di, d in enumerate(max_depths):
                for si, s in enumerate(mss):
                    errors[w, di, si] += sum(_tree_errors(table, per_set[f][w], d, s))
    m_train = len(pos) + len(neg)
    grid = [{"class_importance": _weights_dict(weights[w]), "max_depth": max_depths[di], "min_samples_split": mss[si],
             "cv_errors": int(errors[w, di, si]), "cv_risk": errors[w, di, si] / m_train if m_train else None}
            for w in range(nW) for di in range(len(max_depths)) for si in range(len(mss))]
    w, di, si = _select_cart(errors, max_depths, mss)
    selected = grid[(w * len(max_depths) + di) * len(mss) + si]
    full = trees[k][w]
    model = _truncate(full, max_depths[di], mss[si])
    table = _node_table(full.nodes)

    def metrics(e, a, b):
        fn, fp = _tree_errors(table, per_set[e][w], max_depths[di], mss[si])
        return confusion_metrics(len(a), len(b), fn, fp)

    return SelectionResult("cart", k, ids, grid, selected, model, metrics(k, pos, neg),
                           metrics(k + 1, test_pos, test_neg) if has_test else None,
                           {"fit": t_fit, "eval": t_eval, "total": time.perf_counter() - t_start})


def _weights_dict(ci):
    ci = {0: 1.0, 1: 1.0} if ci is None else ci
    return {str(k): float(v) for k, v in ci.items()}
