"""CPU: k-mer strings to packed k-mers, the grmkm_query_stats layout, the k-mer union and argument errors of
predict_genomes on hand-made fitted models, and the shared output rules of predict / predict_genomes."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from grm_b200 import native
from grm_b200.cart import DecisionTreeClassifier, Node, _tree_output
from grm_b200.learning import kmers_from_strings
from grm_b200.predict import predict_genomes
from grm_b200.scm import KmerRule, SetCoveringMachine, _kmer_string, _scm_output
from oracle import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("k", [1, 5, 11, 21, 31, 32])
def test_kmers_from_strings_round_trips(k):
    rng = np.random.default_rng(k)
    seqs = ["".join(rng.choice(list("ACGT"), size=k)) for _ in range(200)] + ["A" * k, "G" * k]
    x = kmers_from_strings(seqs, k)
    assert x.dtype == np.uint64 and x.shape == (len(seqs),)
    assert [_kmer_string(int(v), k) for v in x] == seqs
    # numpy bytes arrays (kmer_sequences of a .kover file) and bytes give the same
    assert np.array_equal(kmers_from_strings(np.array([s.encode() for s in seqs], dtype=f"S{k}"), k), x)
    assert np.array_equal(kmers_from_strings([s.encode() for s in seqs], k), x)
    # the canonical form of the packed value is the oracle's canonical k-mer
    for s, v in zip(seqs, x):
        v = int(v)
        rc = 0
        for i in range(k):
            rc = (rc << 2) | (((v >> (2 * i)) & 3) ^ 2)
        assert min(v, rc) == oracle.py_canonical(s, k)


def test_kmers_from_strings_lower_case():
    assert np.array_equal(kmers_from_strings(["acgtN"[:4], "AcGt"], 4), kmers_from_strings(["ACGT", "ACGT"], 4))


@pytest.mark.parametrize("seqs,k", [(["ACG"], 4), (["ACGTA"], 4), (["ACGN"], 4), (["AC-T"], 4), (["ACGT", "AC"], 4),
                                    (np.array([b"ACG"], dtype="S4"), 4), (np.array([b"ACGN"], dtype="S4"), 4),
                                    (["ACGT"], 0), (["A" * 33], 33)])
def test_kmers_from_strings_errors(seqs, k):
    with pytest.raises(ValueError):
        kmers_from_strings(seqs, k)


def test_kmers_from_strings_empty():
    assert kmers_from_strings([], 31).shape == (0,)


def test_query_stats_layout_matches_the_header():
    src = open(os.path.join(ROOT, "include", "grmkm.h")).read()
    body = re.search(r"typedef struct grmkm_query_stats \{(.*?)\} grmkm_query_stats;", src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for m in re.finditer(r"(uint32_t|uint64_t|float)\s+([^;]+);", body):
        fields += [(m.group(1), n.strip()) for n in m.group(2).split(",")]
    size = {"uint32_t": 4, "uint64_t": 8, "float": 4}
    ct = native.QueryStats
    assert [f for f, _ in ct._fields_] == [n for _, n in fields]
    for (fname, ftype), (t, _) in zip(ct._fields_, fields):
        assert C.sizeof(ftype) == size[t], fname
    assert C.sizeof(ct) == 8 * 8          # 2 x u32, 6 x u64, a float padded to 8


def test_query_argument_errors_do_not_need_a_device():
    lib = native.load()
    assert lib.grmkm_query(None, None, 0, None, 0, None) == native.E_INVALID


# ---- predict_genomes on hand-made fitted models --------------------------------------------------------------------
class FakeBuilder:
    """Answers query() from a dict genome -> set of canonical k-mers (what grmkm_query computes on the device)."""

    def __init__(self, k, genomes):
        self.k, self.genomes, self.calls = k, genomes, []

    @property
    def query_genome_count(self):
        return len(self.genomes)

    def query(self, kmers):
        self.calls.append(np.asarray(kmers).copy())
        G = len(self.genomes)
        out = np.zeros(((G + 63) // 64, len(kmers)), dtype=np.uint64)
        for i, x in enumerate(kmers):
            can = oracle.py_canonical(_kmer_string(int(x), self.k), self.k)
            for g, have in enumerate(self.genomes):
                if can in have:
                    out[g // 64, i] |= np.uint64(1) << np.uint64(63 - g % 64)
        return out


def can(s):
    return oracle.py_canonical(s, len(s))


def scm(model_type, rules):
    m = SetCoveringMachine(model_type)
    m.model = [KmerRule(i, s, t) for i, (s, t) in enumerate(rules)]
    m.rule_indices = list(range(len(rules)))
    return m


def tree():
    #   node 0: split on AAC  -> present 1, absent 2
    #   node 1: split on CCG  -> present 3 (leaf 1), absent 4 (leaf 0);  node 2: leaf 1
    t = DecisionTreeClassifier()
    t.nodes = [Node(KmerRule(0, "AAC", "presence"), 0.0, 0, 2, 2, 1, 2, 0, np.zeros(0), 1),
               Node(KmerRule(1, "CCG", "presence"), 0.0, 1, 1, 1, 3, 4, 0, np.zeros(0), 1),
               Node(None, 0.0, 1, 1, 0, None, None, 1, np.zeros(0), 0),
               Node(None, 0.0, 2, 1, 0, None, None, 1, np.zeros(0), 0),
               Node(None, 0.0, 2, 0, 1, None, None, 0, np.zeros(0), 0)]
    return t


GENOMES = [{can("AAC"), can("CCG")}, {can("AAC")}, {can("CCG")}, set(), {can("GTT")}]   # GTT = revcomp(AAC)


def test_one_query_for_the_union_of_the_models():
    b = FakeBuilder(3, GENOMES)
    conj = scm("conjunction", [("AAC", "presence"), ("CCG", "presence")])
    disj = scm("disjunction", [("CCG", "absence"), ("TTT", "presence")])
    out = predict_genomes([conj, disj, tree()], b)
    assert len(b.calls) == 1
    assert sorted(_kmer_string(int(x), 3) for x in b.calls[0]) == ["AAC", "CCG", "TTT"]
    assert out[0].tolist() == [1, 0, 0, 0, 0]
    assert out[1].tolist() == [0, 1, 0, 1, 1]
    assert out[2].tolist() == [1, 0, 1, 1, 0]
    assert all(o.dtype == np.uint8 for o in out)
    # the list call equals each model alone
    for m, want in zip([conj, disj, tree()], out):
        assert np.array_equal(predict_genomes([m], FakeBuilder(3, GENOMES))[0], want)


def test_empty_scm_gives_the_constant_of_predict():
    b = FakeBuilder(3, GENOMES)
    assert predict_genomes([scm("conjunction", [])], b)[0].tolist() == [1] * 5
    assert predict_genomes([scm("disjunction", [])], b)[0].tolist() == [0] * 5
    assert b.calls == []


def test_predict_genomes_refusals():
    with pytest.raises(ValueError, match="not fitted"):
        predict_genomes([DecisionTreeClassifier()], FakeBuilder(3, GENOMES))
    with pytest.raises(ValueError, match="3-mers"):
        predict_genomes([scm("conjunction", [("AAC", "presence")])], FakeBuilder(4, GENOMES))
    with pytest.raises(TypeError):
        predict_genomes([object()], FakeBuilder(3, GENOMES))


# ---- the output rules predict and predict_genomes share -------------------------------------------------------------
def test_scm_output_rule():
    cols = np.array([[1, 1], [1, 0], [0, 0]], dtype=np.uint8)
    assert _scm_output("conjunction", cols).tolist() == [1, 0, 0]
    assert _scm_output("disjunction", cols).tolist() == [1, 1, 0]
    assert _scm_output("conjunction", cols[:, :0]).tolist() == [1, 1, 1]
    assert _scm_output("disjunction", cols[:, :0]).tolist() == [0, 0, 0]


def test_tree_output_rule():
    t = tree()
    col = np.array([0, 1, -1, -1, -1])
    cols = np.array([[1, 1], [1, 0], [0, 1], [0, 0]], dtype=np.uint8)
    assert _tree_output(t.nodes, col, cols).tolist() == [1, 0, 1, 1]
    leaf = [Node(None, 0.0, 0, 0, 3, None, None, 0, np.zeros(0), 0)]
    assert _tree_output(leaf, np.array([-1]), np.zeros((3, 0), dtype=np.uint8)).tolist() == [0, 0, 0]


class FakeRC:
    """get_columns over a 0/1 (examples x U) array, absence rules inverted, as KmerRuleClassifications does."""

    def __init__(self, bits):
        self.bits = np.asarray(bits, dtype=np.uint8)

    def get_columns(self, columns):
        U = self.bits.shape[1]
        return np.stack([self.bits[:, c % U] if c < U else 1 - self.bits[:, c % U] for c in columns], axis=1)


def test_predict_runs_the_same_rules():
    rc = FakeRC([[1, 1], [1, 0], [0, 1], [0, 0]])
    t = tree()
    assert t.predict(rc, [0, 1, 2, 3]).tolist() == [1, 0, 1, 1]
    assert t.predict(rc, [3, 0]).tolist() == [1, 1]
    m = scm("conjunction", [("AAC", "presence"), ("CCG", "absence")])
    m.rule_indices = [0, 2 + 1]
    assert m.predict(rc, [0, 1, 2, 3]).tolist() == [0, 1, 0, 0]
    m = scm("disjunction", [])
    assert m.predict(rc, [0, 1]).tolist() == [0, 0]
