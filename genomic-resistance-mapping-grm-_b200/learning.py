"""The learner's hot loop on the GPU-resident matrix -- Python-3 stand-in for
``KmerRuleClassifications`` (bin/kover/core/kover/learning/common/rules.py:96-267) with the same methods,
argument meaning and result types.

The reference streams the packed ``kmer_matrix`` from HDF5 block by block and runs a Cython popcount over it
(popcount.pyx:76-95) for every call of ``sum_rows`` (split risks, split.py:176-188; SCM utilities, scm.py:238-288).
Here the matrix stays where the build left it (HBM) and one kernel does the masked popcount row reduction
(``grmkm_sum_rows``: 8 x ceil(G/64) bytes per k-mer, HBM-bound).  Rule j < U is "k-mer j present", rule U + j
its absence twin (rules.py:146-148, 264).
"""
from __future__ import annotations

import numpy as np

from .create import _minimum_uint_size


def _unpack_binary_bytes_from_ints(a: np.ndarray) -> np.ndarray:
    """(W x n) uint64 -> (64 W x n) 0/1 bytes, genome g = bit 63-(g%64) of word g//64 (kover/utils.py:159-187)."""
    a = np.ascontiguousarray(a, dtype=np.uint64)
    W, n = a.shape
    by = a.astype(">u8").view(np.uint8).reshape(W, n, 8)
    bits = np.unpackbits(by, axis=2)                       # (W, n, 64): bit 63 first
    return np.ascontiguousarray(bits.transpose(0, 2, 1)).reshape(W * 64, n)


class KmerRuleClassifications:
    """Rule classifications of a built matrix.  ``builder`` is a KmerMatrixBuilder (or DistributedBuilder rank)
    whose result is resident; ``n_rows`` the number of genomes (examples)."""

    def __init__(self, builder, n_rows: int):
        self.builder = builder
        self.dataset_initial_n_rows = int(n_rows)
        self.dataset_n_rows = int(n_rows)
        self.dataset_removed_rows: list[int] = []
        self.dataset_removed_rows_mask = np.zeros(self.dataset_initial_n_rows, dtype=bool)
        U, W, _ = builder.dims
        self._U, self._W = int(U), int(W)
        self._matrix = None
        self._kmers = None                 # packed k-mers, fetched once the SCM names a rule (scm.fit_many)

    # -- row bookkeeping (rules.py:171-199): rows are numbered among the rows not removed yet ------------
    def _absolute_rows(self, rows) -> list[int]:
        alive = np.nonzero(~self.dataset_removed_rows_mask)[0]
        return [int(alive[int(r)]) for r in rows]

    def remove_rows(self, rows):
        removed = self._absolute_rows(rows)
        if removed:
            self.dataset_removed_rows = sorted(set(self.dataset_removed_rows + removed))
            self.dataset_removed_rows_mask = np.zeros(self.dataset_initial_n_rows, dtype=bool)
            self.dataset_removed_rows_mask[self.dataset_removed_rows] = True
            self.dataset_n_rows = self.dataset_initial_n_rows - len(self.dataset_removed_rows)

    @property
    def shape(self):
        return self.dataset_n_rows, self._U * 2

    # -- sum_rows (rules.py:201-267) -----------------------------------------------------------------------
    def sum_rows(self, rows):
        """Number of the given rows (no duplicates) each rule classifies as positive: [presence rules | absence rules]."""
        rows = np.asarray(rows)
        result = np.zeros(self._U * 2, dtype=_minimum_uint_size(rows.shape[0]))
        mask = np.zeros(self._W, dtype=np.uint64)
        for idx in self._absolute_rows(np.sort(rows)):
            mask[idx // 64] |= np.uint64(1) << np.uint64(64 - (idx - 64 * (idx // 64)) - 1)      # build_row_mask, rules.py:209-222
        sums = self.builder.sum_rows(mask)
        result[: self._U] = sums
        result[self._U:] = len(rows) - sums.astype(np.int64)
        return result

    # -- get_columns (rules.py:135-171) --------------------------------------------------------------------
    def get_columns(self, columns):
        columns_is_int = False
        if hasattr(columns, "__index__"):
            columns = [columns.__index__()]
            columns_is_int = True
        columns = [int(c) for c in columns]
        invert = np.array([c >= self._U for c in columns])
        cols = np.array([c % self._U if c >= self._U else c for c in columns], dtype=np.int64)
        if self._matrix is None:
            self._matrix = self.builder.matrix()
        row_mask = np.ones(self._W * 64, dtype=bool)
        row_mask[self.dataset_initial_n_rows:] = False
        row_mask[self.dataset_removed_rows] = False
        result = _unpack_binary_bytes_from_ints(self._matrix[:, cols])[row_mask]
        result[:, invert] = 1 - result[:, invert]
        return result.reshape(-1) if columns_is_int else result


_BASE_CODE = np.full(256, 255, dtype=np.uint64)
for _i, _b in enumerate(b"ACTG"):                       # the library's packing: A0 C1 T2 G3, first base most significant
    _BASE_CODE[_b] = _i
    _BASE_CODE[_b | 0x20] = _i                          # lower case: the same base


def kmers_from_strings(seqs, k: int) -> np.ndarray:
    """k-mer strings (str, bytes or a numpy bytes array) -> packed uint64, as ``KmerMatrixBuilder.kmers`` returns
    them (A0 C1 T2 G3, first base most significant).  Upper and lower case are accepted; a string that is not k
    characters long, or a character other than A, C, G, T, raises ValueError."""
    k = int(k)
    if not 1 <= k <= 32:
        raise ValueError(f"k must be in 1..32, not {k}")
    if isinstance(seqs, np.ndarray) and seqs.dtype.kind == "S":
        n = len(seqs)
        if n and (seqs.dtype.itemsize != k or (np.char.str_len(seqs) != k).any()):
            raise ValueError(f"every k-mer must be {k} characters long")
        raw = np.frombuffer(np.ascontiguousarray(seqs).tobytes(), dtype=np.uint8)
    else:
        items = [s.encode("latin-1", "replace") if isinstance(s, str) else bytes(s) for s in seqs]
        n = len(items)
        bad = next((s for s in items if len(s) != k), None)
        if bad is not None:
            raise ValueError(f"every k-mer must be {k} characters long, not {bad!r}")
        raw = np.frombuffer(b"".join(items), dtype=np.uint8)
    codes = _BASE_CODE[raw.reshape(n, k)]
    if (codes == 255).any():
        raise ValueError("a k-mer holds a character other than A, C, G, T")
    kmers = np.zeros(n, dtype=np.uint64)
    for i in range(k):
        kmers = (kmers << np.uint64(2)) | codes[:, i]
    return kmers


def load_kover(path: str, builder) -> KmerRuleClassifications:
    """The k-mer matrix of a ``.kover`` dataset made the resident result of ``builder`` (a KmerMatrixBuilder whose k is
    the dataset's k-mer length), for learning from an existing file.  Reads ``kmer_matrix``, ``kmer_sequences`` and
    ``genome_identifiers`` with hdf5min."""
    from . import hdf5min
    r = hdf5min.H5Reader(path)
    matrix = r["kmer_matrix"].read()
    seqs = r["kmer_sequences"].read()
    n_genomes = len(r["genome_identifiers"].read())
    k = seqs.dtype.itemsize
    if len(seqs) and k != builder.k:
        raise ValueError(f"{path} holds {k}-mers, the builder counts {builder.k}-mers")
    if len(seqs) and not np.isin(np.frombuffer(seqs.tobytes(), dtype=np.uint8), np.frombuffer(b"ACGT", dtype=np.uint8)).all():
        raise ValueError(f"{path}: kmer_sequences holds a character other than A, C, G, T")
    kmers = kmers_from_strings(seqs, k) if len(seqs) else np.zeros(0, dtype=np.uint64)
    builder.load_result(kmers, matrix, n_genomes)
    return KmerRuleClassifications(builder, n_genomes)
