"""Fitted models applied to genomes that were not in the training matrix.

``predict`` of a SetCoveringMachine or a DecisionTreeClassifier reads the rows of the resident matrix.  To classify
new isolates, ``predict_genomes`` needs no matrix of them: a KmerMatrixBuilder holding only their inputs answers one
``query`` for the union of the models' k-mers (a pass over the genomes' packed text on the GPU), and every model's
output rule runs on those columns -- the same rule ``predict`` runs on matrix columns.
"""
from __future__ import annotations

import numpy as np

from .cart import DecisionTreeClassifier, _tree_output
from .learning import _unpack_binary_bytes_from_ints, kmers_from_strings
from .scm import SetCoveringMachine, _scm_output


def _rules(model):
    if isinstance(model, SetCoveringMachine):
        return list(model.model)
    if isinstance(model, DecisionTreeClassifier):
        if not model.nodes:
            raise ValueError("the tree is not fitted")
        return [x.rule for x in model.nodes if x.rule is not None]
    raise TypeError(f"not a fitted SetCoveringMachine or DecisionTreeClassifier: {type(model).__name__}")


def predict_genomes(models, builder) -> list[np.ndarray]:
    """Per model, 0/1 (uint8) per genome row of the inputs ``builder`` holds (rows 0 .. G - 1, G as a build of them
    would have).  One ``builder.query`` for the union of the models' k-mers, whatever the number of models."""
    models = list(models)
    rules = [_rules(m) for m in models]
    union = sorted({r.kmer_sequence for rs in rules for r in rs})
    for s in union:
        if len(s) != builder.k:
            raise ValueError(f"the models hold {len(s)}-mers, the builder counts {builder.k}-mers")
    G = builder.query_genome_count
    if union:
        cols = _unpack_binary_bytes_from_ints(builder.query(kmers_from_strings(union, builder.k)))[:G]
    else:
        cols = np.zeros((G, 0), dtype=np.uint8)
    col_of = {s: i for i, s in enumerate(union)}
    out = []
    for m, rs in zip(models, rules):
        if isinstance(m, SetCoveringMachine):
            c = cols[:, [col_of[r.kmer_sequence] for r in rs]]
            absent = np.array([r.type == "absence" for r in rs], dtype=bool)
            c[:, absent] = 1 - c[:, absent]
            out.append(_scm_output(m.model_type, c))
        else:
            col = np.array([col_of[x.rule.kmer_sequence] if x.rule is not None else -1 for x in m.nodes], dtype=np.int64)
            out.append(_tree_output(m.nodes, col, cols))
    return out
