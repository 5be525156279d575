"""CPU: get_columns and sum_rows of every rule-classification view -- the whole matrix, the pattern view and the column
slices of P ranks over a ThreadExchange -- against a numpy reference over the 0/1 matrix, at W = 3 with a partial last
word, before and after rows are removed."""
import threading

import numpy as np
import pytest

from grm_b200.distributed import ThreadExchange
from grm_b200.learning import KmerRuleClassifications, PatternRuleClassifications, ShardedRuleClassifications
from tests.test_patterns_cpu import FakeBuilder

G, U = 130, 37
REMOVED = [2, 64, 129]


class ContigBuilder(FakeBuilder):
    """FakeBuilder.sum_rows views the words as bytes: the slices and pattern heads it is loaded with are copied first."""

    def load(self, kmers, matrix, G):
        return super().load(kmers, np.ascontiguousarray(matrix), G)


def bits_and_words():
    """A random G x U 0/1 matrix with columns 3 and 17 equal, and its [W][U] words (genome g at bit 63 - g % 64 of
    word g // 64)."""
    rng = np.random.default_rng(7)
    bits = (rng.random((G, U)) < 0.4).astype(np.uint8)
    bits[:, 17] = bits[:, 3]
    W = (G + 63) // 64
    padded = np.zeros((64 * W, U), dtype=np.uint64)
    padded[:G] = bits
    shifts = np.arange(63, -1, -1, dtype=np.uint64)
    words = (padded.reshape(W, 64, U) << shifts[None, :, None]).sum(axis=1, dtype=np.uint64)
    return bits, words


BITS, WORDS = bits_and_words()
COLUMNS = [0, 3, U + 3, 17, U + 17, U + 36, 36, 20, U]
ROWS = [0, 1, 5, 63, 64, 65, 100, 126]


def reference(removed):
    alive = np.setdiff1d(np.arange(G), removed)
    cols = np.array([c % U for c in COLUMNS])
    want_cols = BITS[alive][:, cols]
    want_cols[:, np.array(COLUMNS) >= U] ^= 1
    rows = alive[ROWS]
    present = BITS[rows].sum(axis=0).astype(np.int64)
    return want_cols, np.concatenate([present, len(ROWS) - present])


def check(rc, out):
    """get_columns and sum_rows, then again after remove_rows(REMOVED); the results go to ``out``."""
    for removed in ([], REMOVED):
        if removed:
            rc.remove_rows(removed)
        out.append((rc.get_columns(COLUMNS), rc.get_columns(U + 17), rc.sum_rows(ROWS).astype(np.int64)))


def assert_matches(out):
    assert len(out) == 2
    for (cols, one, sums), removed in zip(out, ([], REMOVED)):
        want_cols, want_sums = reference(removed)
        assert cols.shape == (G - len(removed), len(COLUMNS))
        assert np.array_equal(cols, want_cols)
        assert np.array_equal(one, want_cols[:, 4])
        assert np.array_equal(sums, want_sums)


def whole():
    return KmerRuleClassifications(ContigBuilder().load(np.arange(U, dtype=np.uint64), WORDS, G), G)


def test_the_whole_matrix_view():
    out = []
    check(whole(), out)
    assert_matches(out)


def test_the_pattern_view():
    v = PatternRuleClassifications(whole())
    assert v.n_patterns == U - 1
    out = []
    check(v, out)
    assert_matches(out)


@pytest.mark.parametrize("counts", [[U], [18, U - 18], [0, 1, U - 1]])
def test_sharded_views(counts):
    world = len(counts)
    ends = ThreadExchange.group(world, timeout=20)
    starts = np.concatenate([[0], np.cumsum(counts)])
    outs = [[] for _ in range(world)]
    errors = [None] * world

    def work(r):
        try:
            lo, hi = int(starts[r]), int(starts[r + 1])
            b = ContigBuilder().load(np.arange(lo, hi, dtype=np.uint64), WORDS[:, lo:hi], G)
            check(ShardedRuleClassifications(b, G, r, world, counts, ends[r]), outs[r])
        except BaseException as e:      # noqa: B902
            errors[r] = e

    threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(60)
    assert not any(t.is_alive() for t in threads)
    for e in errors:
        if e is not None:
            raise e
    for out in outs:
        assert_matches(out)
