"""numpy reference of grmkm_patterns: the columns grouped by their bytes (and class), numbered by first column."""
import numpy as np


def reference_patterns(matrix, column_class=None):
    """matrix: (W x U) uint64 -> (pattern_of[U], members[U], member_offsets[P + 1]) as grmkm_patterns returns them."""
    matrix = np.asarray(matrix, dtype=np.uint64)
    W, U = matrix.shape
    keys = np.ascontiguousarray(matrix.T).view(np.uint8).reshape(U, 8 * W)
    cls = np.zeros(U, dtype=np.uint8) if column_class is None else np.asarray(column_class, dtype=np.uint8)
    keys = np.ascontiguousarray(np.concatenate([keys, cls.reshape(U, 1)], axis=1))
    rows = keys.view(np.dtype((np.void, keys.shape[1]))).reshape(U)
    _, first, inverse = np.unique(rows, return_index=True, return_inverse=True)
    rank = np.empty(len(first), dtype=np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(len(first))
    pattern_of = rank[inverse.reshape(-1)]
    members = np.argsort(pattern_of, kind="stable")
    offsets = np.concatenate([[0], np.cumsum(np.bincount(pattern_of, minlength=len(first)))])
    return pattern_of, members, offsets
