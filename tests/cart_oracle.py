"""Reference CART (gini) in plain numpy on unpacked bits, written from the specification of include/grmkm.h
(grmkm_cart_run) and DESIGN.md section 2; it shares nothing with the kernels."""
import numpy as np

from tests.scm_oracle import unpack

LEAF = -1


def _term(a, b, w_pos, w_neg):
    """(A * B) / S of a child with a positives and b negatives, A = w_pos a, B = w_neg b, S = A + B (S > 0 wanted)."""
    A = np.float64(w_pos) * np.asarray(a, dtype=np.float64)
    B = np.float64(w_neg) * np.asarray(b, dtype=np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return (A * B) / (A + B)


def cart_fit(matrix, n_genomes, pos, neg, max_depth=10, min_samples_split=2, w_neg=1.0, w_pos=1.0, blacklist=(),
             equiv_cap=None):
    """-> list of nodes in breadth-first order, each {rule (LEAF for a leaf), score, depth, n_pos, n_neg,
    present_child, absent_child (LEAF for a leaf), prediction, equivalent, equiv_total}.  pos / neg: genome rows;
    max_depth None: no limit; equiv_cap None: record all of T."""
    bits = unpack(matrix, n_genomes).astype(bool)
    U = bits.shape[1]
    allowed = np.ones(U, dtype=bool)
    if len(blacklist):
        allowed[np.asarray(list(blacklist), dtype=np.int64) % U] = False
    P0 = np.zeros(n_genomes, dtype=bool); P0[list(pos)] = True
    N0 = np.zeros(n_genomes, dtype=bool); N0[list(neg)] = True

    nodes, masks = [], {}

    def add(P, N, depth):
        a, b = int(P.sum()), int(N.sum())
        nodes.append({"rule": LEAF, "score": 0.0, "depth": depth, "n_pos": a, "n_neg": b, "present_child": LEAF,
                      "absent_child": LEAF, "prediction": int(np.float64(w_pos) * a > np.float64(w_neg) * b),
                      "equivalent": np.zeros(0, dtype=np.int64), "equiv_total": 0})
        masks[len(nodes) - 1] = (P, N)
        return len(nodes) - 1

    level = [add(P0, N0, 0)]
    while level:
        nxt = []
        for i in level:
            P, N = masks.pop(i)
            nd = nodes[i]
            a, b = nd["n_pos"], nd["n_neg"]
            if (max_depth is not None and nd["depth"] >= max_depth) or a + b < min_samples_split or a == 0 or b == 0:
                continue
            pl = bits[P].sum(axis=0, dtype=np.int64)
            nl = bits[N].sum(axis=0, dtype=np.int64)
            pr, nr = a - pl, b - nl
            ok = allowed & (pl + nl > 0) & (pr + nr > 0)
            if not ok.any():
                continue
            score = _term(pl, nl, w_pos, w_neg) + _term(pr, nr, w_pos, w_neg)
            best = score[ok].min()
            T = np.nonzero(ok & (score == best))[0]
            j = int(T[0])
            nd.update(rule=j, score=float(best), equiv_total=len(T),
                      equivalent=T[: len(T) if equiv_cap is None else equiv_cap].astype(np.int64))
            col = bits[:, j]
            nd["present_child"] = add(P & col, N & col, nd["depth"] + 1)
            nd["absent_child"] = add(P & ~col, N & ~col, nd["depth"] + 1)
            nxt += [nd["present_child"], nd["absent_child"]]
        level = nxt
    return nodes


def cart_predict(nodes, matrix, n_genomes, rows):
    """0/1 per genome row by walking the reference tree."""
    bits = unpack(matrix, n_genomes)
    out = []
    for g in rows:
        i = 0
        while nodes[i]["rule"] != LEAF:
            i = nodes[i]["present_child"] if bits[g, nodes[i]["rule"]] else nodes[i]["absent_child"]
        out.append(nodes[i]["prediction"])
    return np.array(out, dtype=np.uint8)
