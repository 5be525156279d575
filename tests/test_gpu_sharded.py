"""Learning on column slices (-m gpu): a matrix loaded by column ranges into P contexts of one device, driven by P
threads that talk through a ThreadExchange, gives bit for bit what the same calls give on the whole matrix -- SCM
steps, CART nodes, eval_run counts, cross-validated selections and predictions -- for P in {1, 2, 3, 5, 8}, with empty
and one-column slices and cuts through tie sets.  The whole-matrix calls are checked against the numpy references in
test_gpu_scm.py, test_gpu_cart.py and test_gpu_model_selection.py."""
import json
import os
import pickle
import socket
import subprocess
import sys
import threading

import numpy as np
import pytest

from tests import inputs
from tests.test_gpu_scm import loaded, mask, pack, planted

pytestmark = pytest.mark.gpu

ALL = 2**64 - 1


def cuts_for(rng, U, P):
    """P column ranges of [0, U): random cuts, with an empty slice and a one-column slice once P >= 3."""
    inner = sorted(rng.choice(np.arange(1, U), size=P - 1, replace=False).tolist()) if P > 1 else []
    cuts = [0] + inner + [U]
    if P >= 3:
        cuts[1] = 0                         # rank 0 holds nothing
        cuts[2] = 1                         # rank 1 holds column 0 only
        cuts = [0, 0, 1] + sorted(set(c for c in cuts[3:-1] if c > 1)) + [U]
        while len(cuts) < P + 1:
            cuts.insert(-1, cuts[-2])       # further empty slices if the cuts collided
    return cuts


def sharded(matrix, G, cuts, fn, timeout=60.0):
    """fn(rc) on every rank, rank r holding columns [cuts[r], cuts[r + 1]); -> per rank its result or exception."""
    from grm_b200.distributed import ThreadExchange
    from grm_b200.learning import ShardedRuleClassifications
    P = len(cuts) - 1
    ex = ThreadExchange.group(P, timeout=timeout)
    counts = [cuts[r + 1] - cuts[r] for r in range(P)]
    kmers = np.arange(matrix.shape[1], dtype=np.uint64) * np.uint64(7919)
    builders, out = [], [None] * P
    from grm_b200.builder import KmerMatrixBuilder
    for r in range(P):
        b = KmerMatrixBuilder(k=31)
        b.load_result(kmers[cuts[r]:cuts[r + 1]], np.ascontiguousarray(matrix[:, cuts[r]:cuts[r + 1]]), G)
        builders.append(b)
    rcs = [ShardedRuleClassifications(builders[r], G, r, P, counts, ex[r]) for r in range(P)]

    def work(r):
        try:
            out[r] = fn(rcs[r])
        except BaseException as e:      # noqa: B902 -- reported by the caller
            out[r] = e

    threads = [threading.Thread(target=work, args=(r,)) for r in range(P)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout + 60)
    assert not any(t.is_alive() for t in threads), "a rank is still waiting"
    for b in builders:
        b.close()
    return out


def ok(results):
    for r in results:
        if isinstance(r, BaseException):
            raise r
    return results


def same_runs(a, b):
    assert len(a) == len(b)
    for (sa, ea), (sb, eb) in zip(a, b):
        assert sa.tobytes() == sb.tobytes()
        assert np.array_equal(ea, eb)


def scm_jobs(rng, G, labels, W):
    from grm_b200 import native
    jobs = []
    for mt in (native.SCM_CONJUNCTION, native.SCM_DISJUNCTION):
        for p in (0.5, 1.0, 2.5):
            for tb in (True, False):
                sub = rng.random(G) < 0.8
                pos = [g for g in range(G) if labels[g] and sub[g]]
                neg = [g for g in range(G) if not labels[g] and sub[g]]
                jobs.append((mt, p, int(rng.integers(1, 11)), tb, mask(pos, G), mask(neg, G)))
    return jobs


CASES = [(1, 65), (2, 64), (3, 63), (5, 300), (8, 65), (2, 1), (3, 300), (8, 64)]


@pytest.mark.parametrize("P,G", CASES)
def test_scm_on_slices_equals_the_whole_matrix(gpu, P, G):
    rng = np.random.default_rng(100 * P + G)
    U = 700
    bits, labels = planted(rng, G, U, n_copies=6)
    m = pack(bits)
    jobs = scm_jobs(rng, G, labels, m.shape[0])
    cuts = cuts_for(rng, U, P)
    # blacklisted rules owned by different ranks, presence and absence
    bl = np.array(sorted({int(rng.integers(0, 2 * U)) for _ in range(12)} | {cuts[-2], U + cuts[-2]}), dtype=np.uint64)
    with loaded(m, G) as b:
        want = b.scm_run(jobs, bl)
    for got in ok(sharded(m, G, cuts, lambda rc: rc.builder.scm_run(jobs, bl, shard=rc.shard))):
        same_runs(got, want)


@pytest.mark.parametrize("P,G", CASES)
def test_cart_on_slices_equals_the_whole_matrix(gpu, P, G):
    rng = np.random.default_rng(200 * P + G)
    U = 600
    bits, labels = planted(rng, G, U, n_copies=5)
    bits[:, U // 2: U // 2 + 40] = bits[:, [3]]         # a deep tie set the cuts go through
    m = pack(bits)
    pos = [g for g in range(G) if labels[g]]
    neg = [g for g in range(G) if not labels[g]]
    jobs = []
    for cap in (0, 1, 10, ALL):
        for w in ((1.0, 1.0), (0.3, 2.0)):
            for mss in (2, 7):
                jobs.append((int(rng.integers(1, 8)), mss, cap, w[0], w[1], mask(pos, G), mask(neg, G)))
    cuts = cuts_for(rng, U, P)
    bl = np.array([cuts[-2], U + 5], dtype=np.uint64)
    with loaded(m, G) as b:
        want = b.cart_run(jobs, bl)
    for got in ok(sharded(m, G, cuts, lambda rc: rc.builder.cart_run(jobs, bl, shard=rc.shard))):
        same_runs(got, want)


@pytest.mark.parametrize("P,G", [(2, 65), (5, 300), (8, 64)])
def test_eval_run_on_slices_equals_the_whole_matrix(gpu, P, G):
    from grm_b200 import native
    from grm_b200.builder import KmerMatrixBuilder
    rng = np.random.default_rng(300 * P + G)
    U = 500
    bits = (rng.random((G, U)) < 0.4).astype(np.uint8)
    m = pack(bits)
    jobs = []
    for i in range(40):
        sub = rng.random(G)
        pos, neg = mask(np.nonzero(sub < 0.4)[0], G), mask(np.nonzero(sub > 0.6)[0], G)
        if i % 2:
            jobs.append((native.EVAL_SCM, i % 4 // 2, rng.integers(0, 2 * U, size=int(rng.integers(0, 9))), pos, neg))
        else:
            n = 1 + 2 * int(rng.integers(0, 6))           # a chain: node 2 k splits into 2 k + 1 (leaf) and 2 k + 2
            nodes = np.zeros(n, dtype=KmerMatrixBuilder.EVAL_NODE_DTYPE)
            nodes["kmer"] = ALL
            for k in range(0, n - 1, 2):
                nodes[k] = (int(rng.integers(0, U)), k + 1, k + 2)
            jobs.append((native.EVAL_CART, 0, nodes, pos, neg))
    with loaded(m, G) as b:
        want = b.eval_run(jobs)
    for got in ok(sharded(m, G, cuts_for(rng, U, P), lambda rc: rc.builder.eval_run(jobs, shard=rc.shard))):
        assert len(got) == len(want)
        for x, y in zip(got, want):
            assert np.array_equal(x, y)


def selection_json(res):
    d = res.to_dict()
    d.pop("seconds")
    return json.dumps(d, sort_keys=True)


@pytest.mark.parametrize("P", [2, 5])
def test_cross_validation_and_predict_on_slices(gpu, P):
    from grm_b200.cart import DecisionTreeClassifier
    from grm_b200.learning import KmerRuleClassifications
    from grm_b200.model_selection import cross_validate_cart, cross_validate_scm
    from grm_b200.scm import SetCoveringMachine
    rng = np.random.default_rng(40 + P)
    G, U = 150, 3000
    bits, labels = planted(rng, G, U, density=0.4)
    labels = labels ^ (rng.random(G) < 0.15).astype(np.uint8)
    m = pack(bits)
    pos = [g for g in range(120) if labels[g]]
    neg = [g for g in range(120) if not labels[g]]
    tpos = [g for g in range(120, G) if labels[g]]
    tneg = [g for g in range(120, G) if not labels[g]]

    def run(rc):
        a = cross_validate_scm(rc, pos, neg, ["conjunction", "disjunction"], [0.1, 1.0, 5.6], 4, 4, test_pos=tpos,
                               test_neg=tneg, random_seed=3)
        b = cross_validate_cart(rc, pos, neg, [{0: 1.0, 1: 1.0}, {0: 0.5, 1: 2.0}], [1, 2, 4], [2, 10], 3,
                                test_pos=tpos, test_neg=tneg, max_equivalent_rules=5)
        scm = SetCoveringMachine("disjunction", 1.0, 5).fit(rc, pos, neg)
        tree = DecisionTreeClassifier(max_depth=4, max_equivalent_rules=3).fit(rc, pos, neg)
        test = tpos + tneg
        return (selection_json(a), selection_json(b), scm.model, scm.predict(rc, test), tree.nodes,
                tree.predict(rc, test), rc.get_columns([5, U + 7]), rc.sum_rows(test))

    with loaded(m, G) as b:
        want = run(KmerRuleClassifications(b, G))
    for got in ok(sharded(m, G, cuts_for(rng, U, P), run)):
        assert got[0] == want[0] and got[1] == want[1]
        assert got[2] == want[2]
        assert str(got[4]) == str(want[4])
        for i in (3, 5, 6, 7):
            assert np.array_equal(got[i], want[i])


def test_a_tie_list_overflow_on_one_rank_redoes_the_step_everywhere(gpu):
    """1500 identical best columns, all in rank 1's slice: rank 1's tie list (1024 entries at first) overflows, every
    rank grows and redoes the step, and the step lists all of them."""
    from grm_b200 import native
    rng = np.random.default_rng(5)
    G, U = 128, 4000
    bits = (rng.random((G, U)) < 0.3).astype(np.uint8)
    labels = (rng.random(G) < 0.5).astype(np.uint8)
    bits[:, 1000:2500] = labels[:, None]
    m = pack(bits)
    pos = mask(np.nonzero(labels)[0], G)
    neg = mask(np.nonzero(labels == 0)[0], G)
    jobs = [(native.SCM_CONJUNCTION, 1.0, 3, False, pos, neg)]
    with loaded(m, G) as b:
        want = b.scm_run(jobs)
    assert int(want[0][0][0]["equiv_count"]) == 1500
    for got in ok(sharded(m, G, [0, 900, 2600, U], lambda rc: rc.builder.scm_run(jobs, shard=rc.shard))):
        same_runs(got, want)


def test_a_rank_with_a_bad_mask_fails_every_rank(gpu):
    """Rank 1 passes a mask with a bit past the last genome: every rank returns GRMKM_E_INVALID before any device work,
    and no rank is left waiting in an exchange."""
    from grm_b200 import native
    rng = np.random.default_rng(6)
    G, U = 70, 300
    m = pack((rng.random((G, U)) < 0.3).astype(np.uint8))
    good = (native.SCM_CONJUNCTION, 1.0, 3, False, mask([0, 1], G), mask([2, 3], G))
    bad = (native.SCM_CONJUNCTION, 1.0, 3, False, mask([0, 1], G) | mask([G + 1], 128)[:2], mask([2, 3], G))

    def run(rc):
        return rc.builder.scm_run([bad if rc.rank == 1 else good], shard=rc.shard)

    res = sharded(m, G, [0, 100, 200, U], run, timeout=20)
    assert all(isinstance(r, native.GrmkmError) and r.code == native.E_INVALID for r in res), res
    assert "rows >= n_genomes" in str(res[1]) and "rank 1" in str(res[0]) and "rank 1" in str(res[2])


def test_learning_on_the_slices_of_a_two_rank_merge(gpu):
    """The owner slices of a two-rank merge (both ranks emulated in this process): learning on them gives the results
    of the merged whole."""
    import torch
    from grm_b200 import native
    from grm_b200.builder import KmerMatrixBuilder
    from grm_b200.distributed import CudaEngine, ThreadExchange, row_partition, words_per_rank
    from grm_b200.learning import ShardedRuleClassifications
    rng = np.random.default_rng(19)
    world, G = 2, 130
    genomes = [inputs.fasta(rng, n_records=2, max_len=300, shared=[inputs.rand_seq(rng, 2000)]) for _ in range(G)]
    parts, sw = row_partition(G, world), words_per_rank(G, world)
    engines = []
    for r in range(world):
        b = KmerMatrixBuilder(k=19, keep_singletons=True)
        b.set_genome_count(len(parts[r]))
        for i, g in enumerate(parts[r]):
            b.add_genome_bytes(i, genomes[g])
        engines.append(CudaEngine(b))
    bits = max(e.plan_bucket_bits() for e in engines)
    counts, sends = [], []
    for r, e in enumerate(engines):
        e.set_bucket_bits(bits)
        c, s = e.build_partial(world, sw[r])
        counts.append(c); sends.append(s)
    for dst in range(world):
        chunks = []
        for src in range(world):
            width = 1 + sw[src]
            off = sum(counts[src][:dst]) * width
            chunks.append(sends[src][off: off + counts[src][dst] * width])
        engines[dst].merge(torch.cat(chunks), world, dst, [counts[s][dst] for s in range(world)], sw, G)
    owners = [e.b for e in engines]
    allk = np.concatenate([b.kmers() for b in owners])
    allm = np.concatenate([b.matrix() for b in owners], axis=1)
    labels = (rng.random(G) < 0.5)
    pos, neg = mask(np.nonzero(labels)[0], G), mask(np.nonzero(~labels)[0], G)
    sjobs = [(native.SCM_CONJUNCTION, 1.0, 5, True, pos, neg), (native.SCM_DISJUNCTION, 0.5, 5, True, pos, neg)]
    cjobs = [(4, 2, 10, 1.0, 1.0, pos, neg)]
    with KmerMatrixBuilder(k=19) as whole:
        whole.load_result(allk, allm, G)
        want = (whole.scm_run(sjobs), whole.cart_run(cjobs))
    ex = ThreadExchange.group(world)
    col_counts = [int(b.dims[0]) for b in owners]
    rcs = [ShardedRuleClassifications(owners[r], G, r, world, col_counts, ex[r]) for r in range(world)]
    out = [None] * world

    def work(r):
        try:
            out[r] = (owners[r].scm_run(sjobs, shard=rcs[r]), owners[r].cart_run(cjobs, shard=rcs[r]))
        except BaseException as e:      # noqa: B902
            out[r] = e

    threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(120)
    for got in ok(out):
        same_runs(got[0], want[0])
        same_runs(got[1], want[1])
    with pytest.raises(native.GrmkmError) as e:           # the plain call on a slice is still refused
        owners[0].scm_run(sjobs)
    assert e.value.code == native.E_UNSUPPORTED
    for b in owners:
        b.close()


def test_learning_under_torchrun_equals_the_gathered_fit(gpu, tmp_path):
    """Two ranks under a real torch.distributed.run launch: a DistributedBuilder build, then the sharded SCM, CART,
    both CV selections, predict and get_columns on each rank's slice (from_distributed, TorchExchange through the
    ctypes callback), equal on both ranks to rank 0's fit of the gathered matrix (gather() + load_result).  With >= 2
    GPUs the ranks use NCCL; on one GPU they share it and the transport is gloo, as in test_gpu_multi.py."""
    rng = np.random.default_rng(29)
    G = 150
    shared = [inputs.rand_seq(rng, 3000), inputs.rand_seq(rng, 800)]
    genomes = [inputs.fasta(rng, n_records=3, max_len=600, shared=shared) for _ in range(G)]
    labels = (rng.random(G) < 0.5).astype(np.uint8).tolist()
    with open(tmp_path / "genomes.pkl", "wb") as f:
        pickle.dump((genomes, labels), f)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(root, "tests", "_sharded_worker.py"), str(tmp_path), "19"]
    p = subprocess.run(cmd, cwd=root, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-4000:]
    whole = json.loads((tmp_path / "whole.json").read_text())
    assert whole["U"] > 1000 and any(len(m) > 1 for m in whole["scm"])
    for r in range(2):
        got = json.loads((tmp_path / f"sharded_{r}.json").read_text())
        assert len(got["slice"]) == 2 and sum(got["slice"]) == whole["U"] and min(got["slice"]) > 0
        for key in whole:
            assert got[key] == whole[key], (r, key)

