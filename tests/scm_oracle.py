"""Reference Set Covering Machine in plain numpy on unpacked bits, written from the specification of include/grmkm.h
(grmkm_scm_run) and DESIGN.md section 2; it shares nothing with the kernels."""
import numpy as np


def unpack(matrix, n_genomes):
    """(W x U) uint64 words -> (G x U) 0/1 uint8, genome g at bit 63 - g % 64 of word g // 64."""
    matrix = np.asarray(matrix, dtype=np.uint64)
    by = matrix.astype(">u8").view(np.uint8).reshape(matrix.shape[0], matrix.shape[1], 8)
    bits = np.unpackbits(by, axis=2)                           # (W, U, 64), bit 63 first
    return np.ascontiguousarray(bits.transpose(0, 2, 1)).reshape(-1, matrix.shape[1])[:n_genomes]


def scm_fit(matrix, n_genomes, pos, neg, model_type="conjunction", p=1.0, max_rules=10, blacklist=(), tiebreak=True):
    """-> list of steps {rule, utility, positive_errors, negative_covers, equivalent}.  pos / neg: genome rows."""
    bits = unpack(matrix, n_genomes)
    U = bits.shape[1]

    def out(rules):                                          # outputs of rules (< 2U) on every genome, (G, len)
        rules = np.asarray(rules, dtype=np.int64)
        o = bits[:, rules % U]
        return np.where(rules < U, o, 1 - o)

    P0 = np.zeros(n_genomes, dtype=bool); P0[list(pos)] = True
    N0 = np.zeros(n_genomes, dtype=bool); N0[list(neg)] = True
    if model_type == "disjunction":
        P0, N0 = N0, P0
    P, N = P0.copy(), N0.copy()
    allowed = np.ones(2 * U, dtype=bool)
    allowed[np.asarray(list(blacklist), dtype=np.int64)] = False
    steps = []
    while N.sum() > 0 and len(steps) < max_rules:
        # a presence rule outputs 0 where the k-mer is absent, its absence twin where it is present
        inP, inN = bits[P].sum(axis=0, dtype=np.int64), bits[N].sum(axis=0, dtype=np.int64)
        e = np.concatenate([P.sum() - inP, inP])
        c = np.concatenate([N.sum() - inN, inN])
        u = c.astype(np.float64) - np.float64(p) * e.astype(np.float64)      # product rounded, then the difference
        if not allowed.any():
            break
        best = u[allowed].max()
        T = np.nonzero(allowed & (u == best) & ((c > 0) | (e > 0)))[0]
        if len(T) == 0:
            break
        if tiebreak:
            oT = out(T)
            risk = (oT[P0] == 0).sum(axis=0) + (oT[N0] == 1).sum(axis=0)
            T = T[risk == risk.min()]
        r = int(T.min())
        steps.append({"rule": r, "utility": float(best), "positive_errors": int(e[r]), "negative_covers": int(c[r]),
                      "equivalent": T.astype(np.int64)})
        o = out([r])[:, 0]
        P &= o == 1
        N &= o == 1
    return steps
