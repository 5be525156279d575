"""Set Covering Machine on the GPU-resident matrix -- Python-3 stand-in for Kover's learner
(bin/kover/core/kover/learning/learners/scm.py, risk tiebreaker of experiments/experiment_scm.py).

The reference's greedy loop calls ``KmerRuleClassifications.sum_rows`` twice per rule added and works through the 2U
utilities with numpy on the host.  Here every greedy step of a whole batch of fits (model type x p x CV fold) is one
pass over the resident matrix in ``grmkm_scm_run``; only the chosen rules and their equivalent rules come back.

The rule a step chooses is the one the greedy search scored: for a disjunction, the positive and negative examples are
swapped first, so the model itself holds the chosen rules' complements (absence for presence and vice versa) and
predicts 1 when any of them does; a conjunction holds the chosen rules and predicts 1 when all of them do.

A cross-validation or p grid is one ``fit_many`` call; ``model_selection.cross_validate_scm`` scores such a grid on
the held-out examples and picks its hyperparameters.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np

from . import native

KmerRule = namedtuple("KmerRule", "kmer_index kmer_sequence type")     # type: "presence" / "absence"
Iteration = namedtuple("Iteration", "rule utility positive_errors negative_covers equivalent_rules")

_MODEL_TYPES = {"conjunction": native.SCM_CONJUNCTION, "disjunction": native.SCM_DISJUNCTION}


class SetCoveringMachine:
    def __init__(self, model_type: str = "conjunction", p: float = 1.0, max_rules: int = 10):
        if model_type not in _MODEL_TYPES:
            raise ValueError(f"model_type must be 'conjunction' or 'disjunction', not {model_type!r}")
        p = float(p)
        if not (np.isfinite(p) and p >= 0):
            raise ValueError(f"p must be finite and >= 0, not {p}")
        if int(max_rules) < 1:
            raise ValueError("max_rules must be at least 1")
        self.model_type, self.p, self.max_rules = model_type, p, int(max_rules)
        self.model: list[KmerRule] = []
        self.iterations: list[Iteration] = []
        self.rule_indices: list[int] = []         # the model's rules as rule indices (k-mer j present: j, absent: U + j)

    def fit(self, rule_classifications, positive_example_idx, negative_example_idx, rule_blacklist=None,
            tiebreaker="risk"):
        """Learn from the examples (row indices among the rows not removed, as in sum_rows)."""
        fit_many(rule_classifications, [(self, positive_example_idx, negative_example_idx)], rule_blacklist, tiebreaker)
        return self

    def predict(self, rule_classifications, example_idx) -> np.ndarray:
        """0/1 per example (row indices among the rows not removed), from the <= max_rules columns of the model."""
        example_idx = np.asarray(example_idx, dtype=np.int64)
        if not self.rule_indices:
            return _scm_output(self.model_type, np.zeros((len(example_idx), 0), dtype=np.uint8))
        return _scm_output(self.model_type, rule_classifications.get_columns(self.rule_indices)[example_idx])

    def predict_genomes(self, builder) -> np.ndarray:
        """0/1 per genome row of the inputs of ``builder`` (a KmerMatrixBuilder holding genomes that need not have
        been in the training matrix): one ``builder.query`` of the model's k-mers, no build (predict.predict_genomes)."""
        from .predict import predict_genomes
        return predict_genomes([self], builder)[0]


def _scm_output(model_type: str, cols: np.ndarray) -> np.ndarray:
    """The model's output from the 0/1 values of its rules (examples x rules, absence rules already inverted): all of
    them for a conjunction, any of them for a disjunction (an empty model: 1 and 0)."""
    out = cols.all(axis=1) if model_type == "conjunction" else cols.any(axis=1)
    return out.astype(np.uint8)


def _refuse_slices(rule_classifications):
    b = rule_classifications.builder
    if getattr(b, "world", 1) > 1:
        raise ValueError("the matrix is this rank's slice of a multi-GPU build: its best rule is not the answer; "
                         "learn on all slices (learning.ShardedRuleClassifications.from_distributed), or from the "
                         "gathered matrix (DistributedBuilder.gather, then load_result)")


def _row_mask(rule_classifications, idx, W: int) -> np.ndarray:
    rows = np.asarray(rule_classifications._absolute_rows(np.asarray(idx, dtype=np.int64).reshape(-1)), dtype=np.int64)
    mask = np.zeros(W, dtype=np.uint64)
    np.bitwise_or.at(mask, rows // 64, np.left_shift(np.uint64(1), (63 - rows % 64).astype(np.uint64)))
    return mask


def fit_many(rule_classifications, fits, rule_blacklist=None, tiebreaker="risk"):
    """Run every (machine, positive_example_idx, negative_example_idx) of ``fits`` to completion in one batch on the
    GPU (one pass over the matrix per greedy step of all pending fits).  The machines get their model and iterations."""
    _refuse_slices(rule_classifications)
    if tiebreaker not in ("risk", None):
        raise ValueError("tiebreaker must be 'risk' or None")
    rc = rule_classifications
    b = rc.builder
    U, W = rc._U, rc._W
    jobs = []
    for m, pos, neg in fits:
        jobs.append((_MODEL_TYPES[m.model_type], m.p, m.max_rules, tiebreaker == "risk",
                     _row_mask(rc, pos, W), _row_mask(rc, neg, W)))
    blacklist = np.asarray(rule_blacklist if rule_blacklist is not None else [], dtype=np.uint64).reshape(-1)
    results = b.scm_run(jobs, blacklist, shard=rc.shard)
    needed = sorted({int(s["rule"]) % U for _, (steps, _) in zip(fits, results) for s in steps})
    seqs = dict(zip(needed, (_kmer_string(int(x), b.k) for x in rc.kmers_at(needed)))) if needed else {}
    for (m, _, _), (steps, eq) in zip(fits, results):
        m.model, m.iterations, m.rule_indices = [], [], []
        for s in steps:
            r = int(s["rule"])
            o, n = int(s["equiv_offset"]), int(s["equiv_count"])
            m.iterations.append(Iteration(r, float(s["utility"]), int(s["positive_errors"]), int(s["negative_covers"]),
                                          eq[o:o + n].astype(np.int64)))
            mr = r if m.model_type == "conjunction" else (r + U if r < U else r - U)
            j = mr % U
            m.rule_indices.append(mr)
            m.model.append(KmerRule(j, seqs[j], "presence" if mr < U else "absence"))
    return [m for m, _, _ in fits]


def _kmer_string(x: int, k: int) -> str:
    return "".join("ACTG"[(x >> (2 * (k - 1 - i))) & 3] for i in range(k))
