"""Multi-GPU k-mer matrix build: one process per GPU, torch.distributed for the plumbing.

Sharding (SURVEY.md section 8e): genome ROWS are split across ranks in 64-aligned blocks of the
final row order, so a rank's contribution to a column is whole uint64 words.  Each rank runs the
local stages (parse -> extract -> partition -> per-bucket aggregation) and ends with *partial
columns* (hashed k-mer, its local words).  Partial columns are routed to the rank that owns
their hash range with ONE all-to-all (NCCL over NVLink on GPUs; gloo in the CPU tests), and the
owner merges them, applies the singleton filter on the full popcount and orders its slice.
This replaces the hash-routed actor messages of ``mpiexec -n 4 Ray`` (src/app.py:1310).

The compute engine is injectable so the host-side logic can be tested without a GPU
(tests/test_distributed_cpu.py drives it with an oracle-backed engine over gloo).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence

import numpy as np

from . import native
from .native import FASTA


def row_partition(n_genomes: int, world: int) -> list[range]:
    """64-aligned blocks of rows per rank (whole words per rank)."""
    words = (n_genomes + 63) // 64
    out, w0 = [], 0
    for r in range(world):
        nw = words // world + (1 if r < words % world else 0)
        lo, hi = min(64 * w0, n_genomes), min(64 * (w0 + nw), n_genomes)
        out.append(range(lo, hi))
        w0 += nw
    return out


def words_per_rank(n_genomes: int, world: int) -> list[int]:
    words = (n_genomes + 63) // 64
    return [words // world + (1 if r < words % world else 0) for r in range(world)]


def init_process_group_from_env(backend: str | None = None):
    import torch
    import torch.distributed as dist
    if dist.is_initialized():
        return dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29511")
    if backend is None:
        backend = "nccl" if torch.cuda.is_available() else "gloo"
    kw = {}
    if backend == "nccl":
        kw["device_id"] = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    dist.init_process_group(backend=backend, rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]), **kw)
    return dist


class TorchExchange:
    """The all-gather of the sharded runs (learning.ShardedRuleClassifications) over a torch.distributed process group,
    the one the build used by default: the block sizes first, then one all_gather_into_tensor of the blocks padded to
    the largest.  Tensors live on the GPU for NCCL and on the host for gloo, as in DistributedBuilder.slice_counts."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"

    def allgather(self, data: bytes) -> list[bytes]:
        import torch
        import torch.distributed as dist
        sizes = torch.empty(self.world, dtype=torch.int64, device=self.device)
        dist.all_gather_into_tensor(sizes, torch.tensor([len(data)], dtype=torch.int64, device=self.device), group=self.group)
        sizes = sizes.tolist()
        width = max(sizes)
        if width == 0:
            return [b""] * self.world
        mine = torch.zeros(width, dtype=torch.uint8)
        if len(data):
            mine[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8)
        out = torch.empty(self.world * width, dtype=torch.uint8, device=self.device)
        dist.all_gather_into_tensor(out, mine.to(self.device), group=self.group)
        out = out.cpu().numpy()
        return [out[r * width: r * width + sizes[r]].tobytes() for r in range(self.world)]


class ThreadExchange:
    """The all-gather of the sharded runs among `world` threads of one process, each driving its own context (tests,
    or several contexts on one GPU).  ThreadExchange.group(world) makes the ends of all ranks.  A rank that does not
    arrive within `timeout` seconds breaks the barrier: every waiting rank raises TimeoutError instead of hanging."""

    class _Shared:
        def __init__(self, world: int, timeout: float):
            import threading
            self.slots = [b""] * world
            self.barrier = threading.Barrier(world, timeout=timeout)

    def __init__(self, shared: "_Shared", rank: int, world: int):
        self._shared, self.rank, self.world = shared, rank, world

    @classmethod
    def group(cls, world: int, timeout: float = 60.0) -> list["ThreadExchange"]:
        shared = cls._Shared(int(world), float(timeout))
        return [cls(shared, r, int(world)) for r in range(int(world))]

    def _wait(self):
        import threading
        try:
            self._shared.barrier.wait()
        except threading.BrokenBarrierError:
            raise TimeoutError(f"rank {self.rank}: a rank of the thread exchange did not arrive") from None

    def allgather(self, data: bytes) -> list[bytes]:
        self._shared.slots[self.rank] = bytes(data)
        self._wait()                    # every block is in
        out = list(self._shared.slots)
        self._wait()                    # every rank has read them: the slots may be written again
        return out


class HostCounts:
    """The P x P table of partial-column counts, exchanged on the HOST through a file in /dev/shm (the ranks of this
    path share one node, SURVEY.md section 8e): a rank writes its row and then a sequence number, and spins until every
    rank's sequence number has arrived -- microseconds, where ``torch.tensor(counts, device=...)`` + an NCCL all-gather
    + ``.tolist()`` kept the GPU idle for ~0.13 ms between the local aggregate and the export kernel.

    Rows are double-buffered by the parity of the sequence number.  A rank posts build i + 1 only after its
    grmkm_build_partial of build i + 1 has returned, i.e. after its stream -- and with it its merge of build i -- has
    drained, so a post also tells the peers that the poster's receive buffer is free again.
    """

    def __init__(self, dist, world: int, rank: int):
        import mmap
        import tempfile
        self.world, self.rank, self.seq = world, rank, 0
        words = world * 2 * (1 + world)
        name = [None]
        if rank == 0:
            try:
                fd, path = tempfile.mkstemp(prefix="grm_counts_", dir="/dev/shm")
                os.ftruncate(fd, words * 8)
                os.close(fd)
                name[0] = path
            except OSError:
                name[0] = None                                 # no usable /dev/shm: every rank falls back together
        dist.broadcast_object_list(name, src=0)
        if name[0] is None:
            raise OSError("no shared-memory file for the counts table")
        ok = 1
        try:
            with open(name[0], "r+b") as f:
                self._mm = mmap.mmap(f.fileno(), words * 8)
            self.tab = np.frombuffer(self._mm, dtype=np.int64).reshape(world, 2, 1 + world)
        except OSError:
            ok = 0                                             # (a rank that does not see rank 0's /dev/shm: another node)
        flags = [None] * world
        dist.all_gather_object(flags, ok)
        if rank == 0:
            os.unlink(name[0])                                 # the mapping keeps the memory alive
        if not all(flags):
            raise OSError("a rank cannot map the counts table")

    @staticmethod
    def available(world: int) -> bool:
        return (os.path.isdir("/dev/shm") and os.environ.get("GRM_COUNTS", "host") != "nccl"
                and int(os.environ.get("LOCAL_WORLD_SIZE", world)) == world)

    def exchange(self, counts: Sequence[int], timeout_s: float = 120.0) -> list[list[int]]:
        import time
        self.seq += 1
        slot, seq = self.seq & 1, self.seq
        row = self.tab[self.rank, slot]
        row[1:] = counts
        row[0] = seq                                           # (after the counts: x86 keeps the order of the two stores)
        t0 = None
        while True:
            if all(int(self.tab[s, slot, 0]) == seq for s in range(self.world)):
                break
            if t0 is None:
                t0 = time.perf_counter()
            elif time.perf_counter() - t0 > timeout_s:
                raise RuntimeError("a rank did not post its partial-column counts (build %d)" % seq)
        return [[int(x) for x in self.tab[s, slot, 1:]] for s in range(self.world)]


class CudaEngine:
    """Local stages on one GPU through the C ABI (grmkm_build_partial / export / merge)."""

    def __init__(self, builder):
        self.b = builder
        self.launches = 0
        self.local_times, self.local_stats, self.merge_times = {}, {}, {}

    def plan_bucket_bits(self) -> int:
        v = C.c_uint32()
        self.b._check(self.b._lib.grmkm_plan_bucket_bits(self.b._ctx, C.byref(v)))
        return int(v.value)

    def set_bucket_bits(self, bits: int):
        self.b._check(self.b._lib.grmkm_set_bucket_bits(self.b._ctx, int(bits)))

    def build_partial(self, world: int, n_local_words: int, after_counts=None):
        """-> (counts per owner [world], send tensor int64 on the GPU, AoS records of 1+n_local_words).
        after_counts(counts), if given, runs as soon as the counts are known -- before the records are exported, so the
        exchange of the counts overlaps the export kernel."""
        import torch
        counts = (C.c_uint64 * world)()
        self.b._check(self.b._lib.grmkm_build_partial(self.b._ctx, world, counts))
        counts = [int(x) for x in counts]
        if after_counts is not None:
            after_counts(counts)
        st = self.b.stats
        self.launches = st["n_launches"]
        self.local_times = self.b.times
        self.local_stats = st
        n = sum(counts) * (1 + n_local_words)
        send = torch.empty(max(n, 1), dtype=torch.int64, device="cuda")
        self.b._check(self.b._lib.grmkm_export_partials(self.b._ctx, C.c_void_p(send.data_ptr()), send.numel() * 8))
        self.launches += 1
        return counts, send[:n]

    def build_local(self, world: int):
        """Local stages only -> counts per owner [world]; the partial columns stay in the context (export_peers).
        The stage times and statistics are read by collect_local(), once the export is under way (the GPU has nothing to
        do between the local aggregate and the export kernel: no host work belongs there)."""
        counts = (C.c_uint64 * world)()
        self.b._check(self.b._lib.grmkm_build_partial(self.b._ctx, world, counts))
        return [int(x) for x in counts]

    def collect_local(self):
        st = self.b.stats
        self.launches = st["n_launches"]
        self.local_times = self.b.times
        self.local_stats = st

    def export_peers(self, world: int, peer_ptrs: Sequence[int], word_offsets: Sequence[int]):
        """Owner d's slice is stored straight into peer d's receive buffer (asynchronous on the context's stream)."""
        ptrs = (C.c_void_p * world)(*[C.c_void_p(int(p)) for p in peer_ptrs])
        offs = (C.c_uint64 * world)(*[int(o) for o in word_offsets])
        self.b._check(self.b._lib.grmkm_export_partials_peers(self.b._ctx, world, ptrs, offs))

    def merge(self, recv, world: int, rank: int, src_counts: Sequence[int], src_words: Sequence[int], n_genomes: int):
        sc = (C.c_uint64 * world)(*src_counts)
        sw = (C.c_uint32 * world)(*src_words)
        before = self.b.stats["n_launches"]
        self.b._check(self.b._lib.grmkm_merge_partials(self.b._ctx, C.c_void_p(recv.data_ptr() if recv.numel() else 0),
                                                       world, rank, sc, sw, n_genomes))
        self.launches += self.b.stats["n_launches"] - before
        self.merge_times = self.b.times

    def result(self):
        return self.b.kmers(), self.b.matrix()

    def result_host(self):
        return self.b.result_host()


class DistributedBuilder:
    """Same surface as KmerMatrixBuilder, for rank `rank` of `world` processes.

    Rows are LOCAL indices into ``local_rows`` (the global genome rows this rank holds).
    After build(), kmers()/matrix() return this rank's slice of the columns (all word rows);
    gather() assembles the global matrix (ascending hash order, as a one-GPU build) on rank 0.
    """

    def __init__(self, k=31, min_abundance=1, keep_singletons=False, n_genomes=0, rank=0, world=1,
                 input_kind=FASTA, stream=None, device=-1, engine=None, builder=None):
        self.k, self.rank, self.world, self.n_genomes = int(k), int(rank), int(world), int(n_genomes)
        self.local_rows = row_partition(self.n_genomes, self.world)[self.rank]
        self.src_words = words_per_rank(self.n_genomes, self.world)
        self.launches = 0
        self.builder = builder
        self._stream = stream
        if engine is None:
            from .builder import KmerMatrixBuilder
            if stream is None and self.world > 1:
                import torch
                self._stream = stream = torch.cuda.current_stream().cuda_stream      # kernels and collectives on ONE stream
            self.builder = KmerMatrixBuilder(k=k, min_abundance=min_abundance, keep_singletons=keep_singletons,
                                             input_kind=input_kind, device=device, stream=stream)
            if self.world > 1:
                self.builder._check(self.builder._lib.grmkm_set_exchange_rank(self.builder._ctx, self.rank))
            engine = CudaEngine(self.builder)
        self.engine = engine
        self._n_kmers = 0
        # peer exchange (NVLink stores into the owners' receive buffers, torch symmetric memory); None = not tried yet,
        # False = unavailable (other backend, injected engine, GRM_EXCHANGE=nccl): NCCL all-to-all instead
        self._peer = None
        self._peer_buf = None
        self._peer_cap = 0
        self._host_counts = None       # HostCounts once tried; False = not available (several nodes, no /dev/shm, GRM_COUNTS=nccl)

    # -- inputs (local row index) ----------------------------------------------------------------
    def reset(self):
        self.builder.reset()
        self.builder.set_genome_count(len(self.local_rows) if self.world > 1 else self.n_genomes)

    def add_genome_bytes(self, local_row: int, data):
        self.builder.add_genome_bytes(local_row, data)

    def add_genome_device(self, local_row: int, ptr: int, n: int):
        self.builder.add_genome_device(local_row, ptr, n)

    def add_genomes(self, local_rows, data, lens=None, on_device: bool = False):
        self.builder.add_genomes(local_rows, data, lens, on_device)

    def add_genome_files(self, local_row: int, paths):
        self.builder.add_genome_files(local_row, paths)

    # -- build -------------------------------------------------------------------------------------
    def build(self, reuse_partition: bool = False):
        """reuse_partition: keep the bucket count agreed for the previous build of this object instead of agreeing
        again (one all-reduce and a host round trip less).  Collective: every rank passes the same value.  The bucket
        count only sizes the shared-memory tables (a bucket that does not fit is split), never the result."""
        if self.world == 1:
            self.builder.build()
            st = self.builder.stats
            self.launches = st["n_launches"]
            self._n_kmers = st["n_kmers"]
            self.stage_times = self.builder.times
            self.local_stats = st
            return self
        import torch
        import torch.distributed as dist
        dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
        # 1. identical hash partition on every rank
        if not (reuse_partition and getattr(self, "_agreed_bits", None)):
            bits = torch.tensor([self.engine.plan_bucket_bits()], dtype=torch.int64, device=dev)
            dist.all_reduce(bits, op=dist.ReduceOp.MAX)
            self._agreed_bits = int(bits.item())
        self.engine.set_bucket_bits(self._agreed_bits)
        if self._peer is None:
            self._peer = (dev == "cuda" and hasattr(self.engine, "export_peers")
                          and os.environ.get("GRM_EXCHANGE", "peer") != "nccl" and self._peer_probe())
        if self._peer:
            return self._build_peer(torch, dist)
        # 2. local stages -> partial columns grouped by owner
        wl = self.src_words[self.rank]
        ev = None
        if dev == "cuda":
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        # 3. one all-to-all: counts first (sent while the records are still being exported), then the records
        box = {}

        def send_counts(counts):
            if ev:
                ev[0].record()
            c_out = torch.tensor(counts, dtype=torch.int64, device=dev)
            box["c_in"] = torch.empty_like(c_out)
            box["work"] = dist.all_to_all_single(box["c_in"], c_out, async_op=True)

        try:
            counts, send = self.engine.build_partial(self.world, wl, after_counts=send_counts)
        except TypeError:                      # an injected engine without the hook
            counts, send = self.engine.build_partial(self.world, wl)
        if "work" not in box:
            send_counts(counts)
        box["work"].wait()
        src_counts = [int(x) for x in box["c_in"].tolist()]
        in_split = [c * (1 + wl) for c in counts]
        out_split = [src_counts[s] * (1 + self.src_words[s]) for s in range(self.world)]
        if dev == "cpu" and send.is_cuda:
            # CUDA engine under the gloo backend (several ranks sharing one GPU in the tests): the records cross the
            # host for the transport only
            recv_h = torch.empty(sum(out_split), dtype=torch.int64)
            dist.all_to_all_single(recv_h, send.cpu(), output_split_sizes=out_split, input_split_sizes=in_split)
            recv = recv_h.to(send.device)
        else:
            recv = torch.empty(sum(out_split), dtype=torch.int64, device=send.device)
            dist.all_to_all_single(recv, send, output_split_sizes=out_split, input_split_sizes=in_split)
        self.exchange_bytes = int(send.numel() * 8)
        if ev:
            ev[1].record()
        # 4. owner-side merge
        self.engine.merge(recv, self.world, self.rank, src_counts, self.src_words, self.n_genomes)
        lt = dict(getattr(self.engine, "local_times", {}))
        mt = getattr(self.engine, "merge_times", {})
        lt.pop("total", None)
        lt.pop("sort", None)
        if ev:
            ev[1].synchronize()
            lt["exchange"] = ev[0].elapsed_time(ev[1])
        lt.update({"merge_partition": mt.get("scatter", 0.0), "merge_aggregate": mt.get("aggregate", 0.0),
                   "merge_sort": mt.get("sort", 0.0)})
        lt["total"] = sum(lt.values())
        self.stage_times = lt
        self.local_stats = getattr(self.engine, "local_stats", {})
        self.launches = getattr(self.engine, "launches", 0)
        self._recv = recv  # keep alive until the next build
        self._kmers_cache = None
        self._n_kmers = None
        return self

    # -- fused export + exchange over peer memory ---------------------------------------------------
    def _peer_probe(self) -> bool:
        try:
            import torch.distributed._symmetric_memory as sm      # noqa: F401
            return True
        except Exception:
            return False

    def _peer_alloc(self, words: int, torch, dist):
        """(Re)allocate the symmetric receive buffer: collective, every rank calls it with the same size."""
        import torch.distributed._symmetric_memory as sm
        self._peer_buf = sm.empty(int(words), dtype=torch.int64, device=torch.device("cuda", torch.cuda.current_device()))
        self._peer_hdl = sm.rendezvous(self._peer_buf, dist.group.WORLD)
        self._peer_cap = int(words)

    def _build_peer(self, torch, dist):
        """Local stages, then ONE kernel per rank gathers its partial columns and stores every owner's slice straight
        into that owner's receive buffer over NVLink; the ranks meet at a device-side barrier and merge.  The only
        collective besides the barrier is the all-gather of the P x P counts that assigns the offsets."""
        if self._stream and torch.cuda.current_stream().cuda_stream != self._stream:
            # the export kernel and the merge run on the builder's stream: the counts all-gather and the barrier must be
            # ordered on that same stream, whatever stream the caller happens to be on
            with torch.cuda.stream(torch.cuda.ExternalStream(self._stream)):
                return self._build_peer(torch, dist)
        P, r = self.world, self.rank
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        counts = self.engine.build_local(P)
        ev[0].record()
        if self._host_counts is None:
            self._host_counts = False
            if HostCounts.available(P):                                  # (the same answer on every rank: environment only)
                try:
                    self._host_counts = HostCounts(dist, P, r)           # collective; fails on every rank or on none
                except OSError:
                    self._host_counts = False
        if self._host_counts:
            M = self._host_counts.exchange(counts)                       # M[s][d]: columns source s holds for owner d
        else:
            c_out = torch.tensor(counts, dtype=torch.int64, device="cuda")
            c_all = torch.empty(P * P, dtype=torch.int64, device="cuda")
            dist.all_gather_into_tensor(c_all, c_out)
            M = c_all.view(P, P).tolist()
        width = [1 + w for w in self.src_words]
        need = [sum(M[s][d] * width[s] for s in range(P)) for d in range(P)]
        if max(need) > self._peer_cap:                                   # the same decision on every rank (same M)
            self._peer_alloc(max(need) + max(need) // 4 + 1024, torch, dist)
        offs = [sum(M[s][d] * width[s] for s in range(r)) for d in range(P)]
        ev[2].record()                                                   # the counts are agreed (one all-gather, one host round trip)
        self.engine.export_peers(P, list(self._peer_hdl.buffer_ptrs), offs)
        ev[3].record()                                                   # this rank's slices are on their way / have landed
        self._peer_hdl.barrier()                                         # every slice has landed (same stream as the kernel)
        self.engine.collect_local()                                      # (while the export kernel runs)
        self.exchange_bytes = int(sum(counts) * width[r] * 8)
        ev[1].record()
        src_counts = [M[s][r] for s in range(P)]
        self.engine.merge(self._peer_buf[:max(need[r], 1)], P, r, src_counts, self.src_words, self.n_genomes)
        lt = dict(getattr(self.engine, "local_times", {}))
        mt = getattr(self.engine, "merge_times", {})
        lt.pop("total", None)
        lt.pop("sort", None)
        ev[1].synchronize()
        lt["exchange"] = ev[0].elapsed_time(ev[1])
        lt.update({"merge_partition": mt.get("scatter", 0.0), "merge_aggregate": mt.get("aggregate", 0.0),
                   "merge_sort": mt.get("sort", 0.0)})
        lt["total"] = sum(lt.values())
        # where the exchange goes (parts of "exchange", not added to the total again)
        lt["exchange_counts"] = ev[0].elapsed_time(ev[2])
        lt["exchange_export"] = ev[2].elapsed_time(ev[3])
        lt["exchange_barrier"] = ev[3].elapsed_time(ev[1])
        self.stage_times = lt
        self.local_stats = getattr(self.engine, "local_stats", {})
        self.launches = getattr(self.engine, "launches", 0)
        self._kmers_cache = None
        self._n_kmers = None
        return self

    @property
    def n_kmers(self) -> int:
        if self._n_kmers is None:
            self._n_kmers = int(self.builder.dims[0]) if self.builder is not None else len(self.engine.result()[0])
        return self._n_kmers

    def kmers(self):
        return self.engine.result()[0] if self.world > 1 else self.builder.kmers()

    def matrix(self):
        return self.engine.result()[1] if self.world > 1 else self.builder.matrix()

    def result_host(self):
        """This rank's (kmers, matrix) as views of page-locked host memory (valid until the next build)."""
        if self.world > 1 and hasattr(self.engine, "result_host"):
            return self.engine.result_host()
        if self.world > 1:
            return self.engine.result()
        return self.builder.result_host()

    def slice_counts(self) -> list[int]:
        """Columns held by every rank (one all-gather); the global column order is the slices in rank order."""
        if self.world == 1:
            return [self.n_kmers]
        import torch
        import torch.distributed as dist
        dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
        mine = torch.tensor([self.n_kmers], dtype=torch.int64, device=dev)
        out = torch.empty(self.world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(out, mine)
        return [int(x) for x in out.tolist()]

    def write_tsv(self, path: str, names) -> int:
        """Ray Surveyor KmerMatrix.tsv written by all ranks: every rank formats the rows of its own column slice on
        its GPU (k_format_tsv) and writes them at their fixed offset (rows have a constant width).  Returns the
        number of k-mers.  Collective."""
        names = [n if isinstance(n, str) else n.decode() for n in names]
        counts = self.slice_counts()
        hdr = ("kmers" + "".join("\t" + n for n in names) + "\n").encode()
        roww = self.k + 2 * len(names) + 1
        if self.world > 1:
            import torch.distributed as dist
        if self.rank == 0:
            with open(path, "wb") as f:
                f.write(hdr)
                f.truncate(len(hdr) + roww * sum(counts))
        if self.world > 1:
            dist.barrier()
        if counts[self.rank]:
            body = self.builder.tsv(names)[len(hdr):]
            fd = os.open(path, os.O_WRONLY)
            try:
                off, view = len(hdr) + roww * sum(counts[:self.rank]), memoryview(body)
                while len(view):
                    n = os.pwrite(fd, view[:1 << 30], off)
                    off += n
                    view = view[n:]
            finally:
                os.close(fd)
        if self.world > 1:
            dist.barrier()
        return sum(counts)

    def gather(self):
        """Global (kmers, matrix [W][U]) in ascending hash order on rank 0, None elsewhere."""
        km, mat = self.kmers(), self.matrix()
        if self.world == 1:
            return km, mat
        import torch.distributed as dist
        objs = [None] * self.world if self.rank == 0 else None
        dist.gather_object((km, mat), objs, dst=0)
        if self.rank != 0:
            return None
        # rank r owns the r-th contiguous range of the hash space and its slice is in ascending hash order, so
        # the concatenation in rank order IS the global column order -- the same bytes as a one-GPU build
        allk = np.concatenate([o[0] for o in objs])
        allm = np.concatenate([o[1] for o in objs], axis=1)
        return allk, np.ascontiguousarray(allm)

    def close(self):
        if self.builder is not None:
            self.builder.close()
