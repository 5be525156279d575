"""Sharded learning, host side (no GPU): the exchanges (ThreadExchange, TorchExchange on gloo), the map of global
columns to their owners, and the checks of ShardedRuleClassifications."""
import os
import socket
import subprocess
import sys
import threading

import numpy as np
import pytest

from grm_b200.distributed import ThreadExchange
from grm_b200.learning import ShardedRuleClassifications, column_owners

HERE = os.path.dirname(os.path.abspath(__file__))


def blocks_of(rank, rnd):
    """Rank `rank`'s block in round `rnd`: sizes vary by rank and round, some are empty."""
    return bytes([(rank * 7 + rnd + i) % 256 for i in range((rank * 5 + rnd * 3) % 11)])


def run_threads(world, fn):
    out = [None] * world
    ends = ThreadExchange.group(world, timeout=5)

    def work(r):
        try:
            out[r] = fn(ends[r], r)
        except BaseException as e:      # noqa: B902
            out[r] = e

    threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(30)
    assert not any(t.is_alive() for t in threads)
    return out


@pytest.mark.parametrize("world", [1, 2, 3, 5])
def test_thread_exchange_gathers_in_rank_order(world):
    def fn(ex, r):
        return [ex.allgather(blocks_of(r, rnd)) for rnd in range(6)]
    for got in run_threads(world, fn):
        assert got == [[blocks_of(q, rnd) for q in range(world)] for rnd in range(6)]


def test_thread_exchange_times_out_instead_of_hanging():
    def fn(ex, r):
        if r == 2:
            return "absent"
        return ex.allgather(b"x")
    out = run_threads(3, fn)
    assert isinstance(out[0], TimeoutError) and isinstance(out[1], TimeoutError) and out[2] == "absent"


def free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


WORKER = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from grm_b200.distributed import TorchExchange, init_process_group_from_env
from tests.test_sharded_cpu import blocks_of
init_process_group_from_env("gloo")
ex = TorchExchange()
world = ex.world
for rnd in range(6):
    got = ex.allgather(blocks_of(ex.rank, rnd))
    assert got == [blocks_of(q, rnd) for q in range(world)], (rnd, got)
assert ex.allgather(b"") == [b""] * world
dist.barrier()
dist.destroy_process_group()
"""


@pytest.mark.parametrize("world", [2, 3])
def test_torch_exchange_on_gloo(world):
    root = os.path.dirname(HERE)
    port = free_port()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen([sys.executable, "-c", WORKER, root], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, cwd=root))
    for p in procs:
        out, _ = p.communicate(timeout=240)
        assert p.returncode == 0, out.decode()[-2000:]


TIMEOUT_WORKER = r"""
import datetime, os, sys, time
sys.path.insert(0, sys.argv[1])
import torch.distributed as dist
from grm_b200.distributed import TorchExchange
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]),
                        timeout=datetime.timedelta(seconds=3))
ex = TorchExchange()
assert ex.allgather(b"ab") == [b"ab", b"ab"]
if ex.rank == 1:
    time.sleep(12)                      # never joins the second all-gather
    sys.exit(0)
t0 = time.time()
try:
    ex.allgather(b"x")
except Exception:
    assert time.time() - t0 < 11, time.time() - t0
    print("timed out", flush=True)
    os._exit(0)                         # the group is unusable after a timeout: no clean shutdown
sys.exit("the all-gather returned without rank 1")
"""


def test_torch_exchange_times_out_instead_of_hanging():
    """A rank that never joins: the other's TorchExchange raises when the process group's timeout expires."""
    root = os.path.dirname(HERE)
    port = free_port()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen([sys.executable, "-c", TIMEOUT_WORKER, root], env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.STDOUT, cwd=root))
    outs = []
    for p in procs:
        out, _ = p.communicate(timeout=120)
        outs.append(out.decode())
        assert p.returncode == 0, out.decode()[-2000:]
    assert "timed out" in outs[0]


def test_column_owners_maps_global_columns_to_slices():
    counts = [0, 1, 4, 0, 3]                        # an empty first slice, a one-column slice, an empty middle one
    owner, local = column_owners(counts, range(8))
    assert owner.tolist() == [1, 2, 2, 2, 2, 4, 4, 4]
    assert local.tolist() == [0, 0, 1, 2, 3, 0, 1, 2]
    o, l_ = column_owners(counts, [])
    assert len(o) == len(l_) == 0
    with pytest.raises(IndexError):
        column_owners(counts, [8])


def test_absence_rules_map_to_their_columns():
    """A sharded rule classification counts U as the sum of the slices: rule U + j is the absence twin of column j."""
    class Slice:
        dims = (4, 1, 10)
    rc = ShardedRuleClassifications(Slice(), 10, 1, 3, [2, 4, 3], exchange=None)
    assert (rc.col_offset, rc.n_kmers_total, rc.shape) == (2, 9, (10, 18))
    owner, local = column_owners(rc.col_counts, [r % rc._U for r in (3, 9 + 3, 9 + 8)])
    assert owner.tolist() == [1, 1, 2] and local.tolist() == [1, 1, 2]
    assert rc.shard is rc


@pytest.mark.parametrize("counts", [[2, 5, 3], [2, 4], [-1, 5, 5]])
def test_col_counts_that_do_not_fit_the_slice_are_refused(counts):
    class Slice:
        dims = (4, 1, 10)
    with pytest.raises(ValueError):
        ShardedRuleClassifications(Slice(), 10, 1, 3, counts, exchange=None)


def test_the_plain_rule_classifications_has_no_shard():
    from grm_b200.learning import KmerRuleClassifications
    assert KmerRuleClassifications.shard is None
