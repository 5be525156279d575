"""Reference of grmkm_eval_run in plain numpy on unpacked bits, written from include/grmkm.h; it shares nothing with
the kernels.  bits: (G x U) 0/1; pos / neg: genome rows."""
import numpy as np

LEAF = None


def eval_scm(bits, model_type, rules, pos, neg):
    """(R + 1, 2): per prefix of r rules, (#pos the model outputs 0 on, #neg it outputs 1 on)."""
    G, U = bits.shape
    out = np.full(G, model_type == "conjunction", dtype=bool)
    res = []
    for r in range(len(rules) + 1):
        res.append((int((~out[list(pos)]).sum()), int(out[list(neg)].sum())))
        if r < len(rules):
            rule = int(rules[r])
            col = bits[:, rule % U].astype(bool) ^ (rule >= U)
            out = out & col if model_type == "conjunction" else out | col
    return np.array(res, dtype=np.int64).reshape(-1, 2)


def eval_cart(bits, nodes, pos, neg):
    """(n, 2): per node, (#pos, #neg) examples that reach it.  nodes: (kmer or LEAF, present_child, absent_child)."""
    res = np.zeros((len(nodes), 2), dtype=np.int64)
    for c, rows in enumerate((pos, neg)):
        for g in rows:
            i = 0
            while True:
                res[i, c] += 1
                kmer, present, absent = nodes[i]
                if kmer is LEAF:
                    break
                i = present if bits[g, kmer] else absent
    return res
