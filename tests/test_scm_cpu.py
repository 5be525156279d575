"""CPU: the Set Covering Machine's numpy reference on hand-computed cases, the layouts of the new ABI structs, and the
argument errors that need no device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from grm_b200 import native
from tests.scm_oracle import scm_fit

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# genomes g0..g3 (rows) x k-mers k0..k4 (columns); rule r < 5: k-mer r present, rule 5 + r: absent
BITS = np.array([[0, 1, 0, 1, 0],
                 [1, 1, 1, 1, 0],
                 [0, 0, 1, 0, 0],
                 [0, 0, 1, 1, 1]])


def packed(bits):
    G, U = bits.shape
    m = np.zeros(((G + 63) // 64, U), dtype=np.uint64)
    for g in range(G):
        m[g // 64] |= bits[g].astype(np.uint64) << np.uint64(63 - g % 64)
    return m


def steps(**kw):
    args = dict(model_type="conjunction", p=1.0, max_rules=10, blacklist=(), tiebreak=True, pos=[0, 1], neg=[2, 3])
    args.update(kw)
    got = scm_fit(packed(BITS), 4, **args)
    return [(s["rule"], s["utility"], s["positive_errors"], s["negative_covers"], s["equivalent"].tolist()) for s in got]


def test_conjunction():
    # p = 1: u = c - e; k1 present is 1 on both positives and 0 on both negatives: u = 2, alone
    assert steps() == [(1, 2.0, 0, 2, [1])]


def test_tie_broken_by_risk():
    # p = 0: u = c; c = 2 for k0 (e = 1), k1 (e = 0) and "k2 absent" (e = 1).  risk = e + #N0 the rule outputs 1 on:
    # 1, 0, 1 -> the tiebreaker keeps k1 only; without it the lowest index of the three wins
    assert steps(p=0.0, tiebreak=False) == [(0, 2.0, 1, 2, [0, 1, 7])]
    assert steps(p=0.0) == [(1, 2.0, 0, 2, [1])]


def test_disjunction_swaps_the_examples():
    # P = {g2, g3}, N = {g0, g1}: "k1 absent" is 1 on g2, g3 and 0 on g0, g1
    assert steps(model_type="disjunction") == [(6, 2.0, 0, 2, [6])]


def test_rules_that_change_nothing_are_never_chosen():
    # P = {g1}, N = {g3}, k0, k1 present and k4 absent blacklisted: u* = 0, held by k2 and k3 present (1 on both
    # examples: they change nothing) and by "k2 absent", "k3 absent" (e = 1, c = 1)
    assert steps(pos=[1], neg=[3], blacklist=[0, 1, 9]) == [(7, 0.0, 1, 1, [7, 8])]


def test_stop_on_empty_tie_set():
    # the same with both absence rules blacklisted too: only the rules that change nothing reach u* = 0
    assert steps(pos=[1], neg=[3], blacklist=[0, 1, 7, 8, 9]) == []


def test_blacklist_and_stop_on_max_rules():
    # without k0, k1 present and "k2 absent": k3 present and "k4 absent" tie at u = 1 (same risk); k3 present leaves
    # N = {g3}, which "k4 absent" covers next
    assert steps(blacklist=[0, 1, 7]) == [(3, 1.0, 0, 1, [3, 9]), (9, 1.0, 0, 1, [9])]
    assert steps(blacklist=[0, 1, 7], max_rules=1) == [(3, 1.0, 0, 1, [3, 9])]


def test_stop_on_empty_negatives():
    assert steps(neg=[]) == []


def _header_struct(name):
    src = open(os.path.join(ROOT, "include", "grmkm.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return [(m.group(1).strip(), m.group(2)) for m in re.finditer(r"([A-Za-z_0-9 *]+?)\s*\b(\w+);", body)]


@pytest.mark.parametrize("name,cls", [("grmkm_scm_job", "ScmJob"), ("grmkm_scm_step", "ScmStep")])
def test_struct_layouts_match_the_header(name, cls):
    size = {"uint32_t": 4, "uint64_t": 8, "double": 8, "const uint64_t*": 8}
    fields = _header_struct(name)
    ct = getattr(native, cls)
    assert [f for f, _ in ct._fields_] == [n for _, n in fields]
    for (fname, ftype), (t, _) in zip(ct._fields_, fields):
        assert C.sizeof(ftype) == size[t], fname
    assert C.sizeof(ct) == sum(size[t] for t, _ in fields)


def test_argument_errors_do_not_need_a_device():
    lib = native.load()
    job = native.ScmJob(C.sizeof(native.ScmJob), 0, 1, 1, 1.0, None, None)
    assert lib.grmkm_scm_run(None, 1, C.byref(job), None, 0) == native.E_INVALID
    assert lib.grmkm_scm_run(None, 0, None, None, 0) == native.E_INVALID
    n = C.c_uint64()
    assert lib.grmkm_scm_result(None, 0, None, 0, C.byref(n), None, 0, C.byref(n)) == native.E_INVALID
    assert lib.grmkm_load_result(None, None, None, 0, 1) == native.E_INVALID


@pytest.mark.parametrize("kw", [dict(model_type="dnf"), dict(p=-1.0), dict(p=float("nan")), dict(p=float("inf")),
                                dict(max_rules=0)])
def test_machine_arguments(kw):
    from grm_b200.scm import SetCoveringMachine
    with pytest.raises(ValueError):
        SetCoveringMachine(**kw)


def test_a_multi_gpu_slice_is_refused():
    from grm_b200.distributed import DistributedBuilder
    from grm_b200.learning import KmerRuleClassifications
    from grm_b200.scm import SetCoveringMachine
    rc = KmerRuleClassifications.__new__(KmerRuleClassifications)
    rc.builder = DistributedBuilder(n_genomes=128, rank=0, world=2, engine=object())
    with pytest.raises(ValueError, match="slice"):
        SetCoveringMachine().fit(rc, [0], [1])
