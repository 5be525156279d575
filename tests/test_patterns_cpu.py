"""CPU: the numpy reference of grmkm_patterns, PatternRuleClassifications' mapping between patterns and columns on a
fake builder (tie sets expanded, CART lists capped, blacklists that split a pattern, refusals), and the binding of
grmkm_patterns against include/grmkm.h."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from grm_b200 import native
from grm_b200.learning import KmerRuleClassifications, PatternRuleClassifications, ShardedRuleClassifications
from tests.pattern_oracle import reference_patterns

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL = 2**64 - 1


class FakeBuilder:
    """A builder whose 'device' is numpy: patterns from the reference, learner runs answered from canned results."""

    def __init__(self, k=31, device=-1):
        self.k, self.device = k, device
        self.kmers_ = np.zeros(0, dtype=np.uint64)
        self.matrix_ = np.zeros((1, 0), dtype=np.uint64)
        self.G = 64
        self.canned, self.calls = None, []

    def load(self, kmers, matrix, G):
        self.kmers_, self.matrix_, self.G = np.asarray(kmers, dtype=np.uint64), np.asarray(matrix, dtype=np.uint64), G
        return self

    @property
    def dims(self):
        return self.matrix_.shape[1], self.matrix_.shape[0], self.G

    def patterns(self, dst, column_class=None):
        po, mem, off = reference_patterns(self.matrix_, column_class)
        heads = mem[off[:-1]]
        dst.load(self.kmers_[heads], self.matrix_[:, heads], self.G)
        self.calls.append(("patterns", column_class))
        return po.astype(np.uint32), mem.astype(np.uint32), off.astype(np.uint64)

    def kmers(self):
        return self.kmers_

    def matrix(self):
        return self.matrix_

    def columns(self, idx):
        return self.matrix_[:, np.asarray(idx, dtype=np.int64)]

    def sum_rows(self, mask):
        x = self.matrix_ & np.asarray(mask, dtype=np.uint64)[:, None]
        return np.unpackbits(x.view(np.uint8).reshape(x.shape + (8,)), axis=2).sum(axis=(0, 2)).astype(np.uint32)

    def scm_run(self, jobs, blacklist=(), shard=None):
        self.calls.append(("scm_run", np.asarray(blacklist, dtype=np.uint64)))
        return self.canned

    def cart_run(self, jobs, blacklist=(), shard=None):
        self.calls.append(("cart_run", np.asarray(blacklist, dtype=np.uint64)))
        return self.canned

    def eval_run(self, jobs, shard=None):
        self.calls.append(("eval_run", jobs))
        return self.canned


def words(bits):
    """(G <= 64) x U 0/1 -> 1 x U words."""
    bits = np.asarray(bits, dtype=np.uint64)
    return (bits << np.arange(63, 63 - bits.shape[0], -1, dtype=np.uint64)[:, None]).sum(axis=0, dtype=np.uint64)[None, :]


def view_of(cols, blacklist=None):
    """cols: one small integer per column, its presence word."""
    m = np.asarray(cols, dtype=np.uint64)[None, :]
    b = FakeBuilder().load(np.arange(m.shape[1], dtype=np.uint64) * np.uint64(3), m, 64)
    rc = KmerRuleClassifications(b, 64)
    return rc, PatternRuleClassifications(rc, blacklist)


def test_reference_numbers_patterns_by_first_column():
    m = np.array([[7, 9, 7, 8, 9, 7]], dtype=np.uint64)
    po, mem, off = reference_patterns(m)
    assert po.tolist() == [0, 1, 0, 2, 1, 0]
    assert mem.tolist() == [0, 2, 5, 1, 4, 3] and off.tolist() == [0, 3, 5, 6]
    po, mem, off = reference_patterns(m, [0, 0, 2, 0, 0, 0])          # a class splits pattern 0
    assert po.tolist() == [0, 1, 2, 3, 1, 0] and off.tolist() == [0, 2, 4, 5, 6]
    assert reference_patterns(np.zeros((0, 3), dtype=np.uint64))[0].tolist() == [0, 0, 0]    # no genomes: one pattern
    assert reference_patterns(np.zeros((2, 0), dtype=np.uint64))[2].tolist() == [0]


def test_the_view_maps_patterns_and_columns():
    rc, v = view_of([5, 6, 5, 7, 6, 5, 8])
    U, P = 7, 4
    assert (v._U, v.n_patterns) == (U, P)
    assert v.pattern_of.tolist() == [0, 1, 0, 2, 1, 0, 3] and v.heads.tolist() == [0, 1, 3, 6]
    assert v.members_of([2, 0]).tolist() == [3, 0, 2, 5]
    assert v.expand_rules([0, P + 1]).tolist() == [0, 2, 5, U + 1, U + 4]
    assert v.rule_of_pattern([1, P + 2]).tolist() == [1, U + 3]
    assert v.pattern_rules([5, U + 4]).tolist() == [0, P + 1]
    assert np.array_equal(v.builder.sum_rows(np.array([~np.uint64(0)])), rc.builder.sum_rows(np.array([~np.uint64(0)])))
    assert np.array_equal(v.get_columns([4, U + 2]), rc.get_columns([4, U + 2]))
    assert np.array_equal(v.sum_rows([0, 3, 60]), rc.sum_rows([0, 3, 60]))
    assert np.array_equal(v.kmers_at([4, 2]), rc.kmers_at([4, 2]))


def test_scm_steps_come_back_as_columns_with_complete_sorted_ties():
    rc, v = view_of([5, 6, 5, 7, 6, 5, 8])
    U, P = 7, 4
    steps = np.zeros(2, dtype=[("rule", np.uint64), ("utility", np.float64), ("positive_errors", np.uint32),
                               ("negative_covers", np.uint32), ("equiv_offset", np.uint64), ("equiv_count", np.uint64)])
    steps[0] = (P + 1, 2.5, 1, 3, 0, 2)
    steps[1] = (2, 1.0, 0, 1, 2, 1)
    v.pattern_builder.canned = [(steps, np.array([1, P + 1, 2], dtype=np.uint64))]
    (got, eq), = v.builder.scm_run([None])
    assert got["rule"].tolist() == [U + 1, 3]
    assert got["equiv_offset"].tolist() == [0, 4] and got["equiv_count"].tolist() == [4, 1]
    assert eq.tolist() == [1, 4, U + 1, U + 4, 3]
    assert got["utility"].tolist() == [2.5, 1.0]


def cart_nodes(rows):
    from grm_b200.builder import KmerMatrixBuilder
    nodes = np.zeros(len(rows), dtype=KmerMatrixBuilder.CART_NODE_DTYPE)
    for i, (rule, off, cnt, total, pc) in enumerate(rows):
        nodes[i] = (rule, 0.25, 0, 3, 4, pc, pc + 1 if pc != 0xFFFFFFFF else pc, 1, off, cnt, total)
    return nodes


def test_cart_ties_are_capped_over_members_not_patterns():
    """The cap counter-example: pattern 0 holds columns {0, 8}, pattern 1 holds {1, 9}; with equiv_cap = 2 the library
    records the two smallest tie patterns, and the view keeps the two smallest members, 0 and 1."""
    rc, v = view_of([5, 6, 7, 8, 9, 10, 11, 12, 5, 6])
    leaf = 0xFFFFFFFF
    v.pattern_builder.canned = [(cart_nodes([(1, 0, 2, 4, 1), (ALL, 2, 0, 0, leaf), (ALL, 2, 0, 0, leaf)]),
                                 np.array([0, 1], dtype=np.uint64))]
    for cap, want in ((2, [0, 1]), (1, [0]), (0, []), (ALL, [0, 1, 8, 9])):
        (nodes, eq), = v.builder.cart_run([(3, 2, cap, 1.0, 1.0, None, None)])
        assert int(nodes[0]["rule"]) == 1 and int(nodes[0]["equiv_total"]) == 4
        assert int(nodes[0]["equiv_count"]) == len(want) and eq.tolist() == want
        assert int(nodes[1]["rule"]) == ALL and nodes["equiv_offset"].tolist() == [0, len(want), len(want)]


def test_a_blacklist_that_splits_a_pattern():
    # columns 0, 2, 5 share a vector; 2 is presence-blacklisted, 5 absence-blacklisted
    U = 7
    rc, v = view_of([5, 6, 5, 7, 6, 5, 8], [2, U + 5, U + 6])
    P = v.n_patterns
    assert len({int(v.pattern_of[j]) for j in (0, 2, 5)}) == 3
    assert P == 6
    assert sorted(v.pattern_blacklist.tolist()) == sorted([int(v.pattern_of[2]), P + int(v.pattern_of[5]),
                                                           P + int(v.pattern_of[6])])
    cls = rc.builder.calls[-1][1]
    assert cls.tolist() == [0, 0, 1, 0, 0, 2, 2]
    v.pattern_builder.canned = []
    v.builder.scm_run([], [U + 6, 2, U + 5])
    assert np.array_equal(v.pattern_builder.calls[-1][1], v.pattern_blacklist)
    with pytest.raises(ValueError, match="build a PatternRuleClassifications"):
        v.builder.cart_run([], [2])
    with pytest.raises(ValueError, match="build a PatternRuleClassifications"):
        v.builder.scm_run([], None)


def test_eval_jobs_are_mapped_to_patterns():
    from grm_b200.builder import KmerMatrixBuilder
    rc, v = view_of([5, 6, 5, 7, 6, 5, 8])
    U, P = 7, 4
    nodes = np.zeros(3, dtype=KmerMatrixBuilder.EVAL_NODE_DTYPE)
    nodes[0] = (4, 1, 2)
    nodes[1] = (ALL, 0, 0)
    nodes[2] = (ALL, 0, 0)
    v.pattern_builder.canned = ["counts"]
    assert v.builder.eval_run([(native.EVAL_SCM, 0, [5, U + 3, U + 6], None, None),
                               (native.EVAL_CART, 0, nodes, None, None)]) == ["counts"]
    jobs = v.pattern_builder.calls[-1][1]
    assert jobs[0][2].tolist() == [0, P + 2, P + 3]
    assert jobs[1][2]["kmer"].tolist() == [1, ALL, ALL]
    assert nodes["kmer"].tolist() == [4, ALL, ALL]                  # the caller's nodes are left as they are


def test_views_of_slices_and_of_views_are_refused():
    b = FakeBuilder().load(np.zeros(3, dtype=np.uint64), np.ones((1, 3), dtype=np.uint64), 64)
    with pytest.raises(ValueError, match="slices"):
        PatternRuleClassifications(ShardedRuleClassifications(b, 64, 0, 1, [3], None))
    rc = KmerRuleClassifications(b, 64)
    with pytest.raises(ValueError):
        PatternRuleClassifications(PatternRuleClassifications(rc))
    with pytest.raises(ValueError, match="2 x 3"):
        PatternRuleClassifications(rc, [6])


def test_binding_matches_the_header():
    src = open(os.path.join(ROOT, "include", "grmkm.h")).read()
    body = re.search(r"typedef struct grmkm_pattern_stats \{(.*?)\} grmkm_pattern_stats;", src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = [f for decl in body.split(";") if decl.strip() for f in re.findall(r"(\w+)\s*(?:,|$)", decl.strip())]
    assert fields == [n for n, _ in native.PatternStats._fields_]
    assert C.sizeof(native.PatternStats) == 24
    proto = re.search(r"int grmkm_patterns\((.*?)\);", src, re.S).group(1)
    assert len(proto.split(",")) == 10
    lib = native.load()
    assert len(lib.grmkm_patterns.argtypes) == 10
    assert native.ABI_VERSION == 16


def test_patterns_argument_errors_do_not_need_a_device():
    lib = native.load()
    assert lib.grmkm_patterns(None, None, None, None, 0, None, 0, None, 0, None) == native.E_INVALID
