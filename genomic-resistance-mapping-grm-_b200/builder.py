"""KmerMatrixBuilder -- numpy-facing wrapper over the C ABI (one context = one GPU).

Stands where the reference shells out to ``multidsk`` + ``dsk2kover``
(bin/kover/core/kover/dataset/tools/kmer_count.py:23-53, kmer_pack.py:23-39) and to
``Ray`` (src/app.py:1310): same parameters, result as arrays instead of temp files.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Sequence

import numpy as np

from . import native
from .native import FASTA, FASTQ, GrmkmError  # noqa: F401


class KmerMatrixBuilder:
    def __init__(self, k: int = 31, min_abundance: int = 1, keep_singletons: bool = False,
                 input_kind: int = FASTA, device: int = -1, bucket_bits: int = 0, flags: int = 0,
                 stream: int | None = None):
        self._lib = native.load()
        self._ctx = C.c_void_p()
        self._keep = []          # borrowed host buffers must outlive build()
        self._rows = 0           # max genome row + 1 of the inputs added since the last reset
        self._declared = 0       # set_genome_count
        self.k = int(k)
        self.device = int(device)
        cfg = native.Config(C.sizeof(native.Config), int(k), int(min_abundance), int(bool(keep_singletons)),
                            int(input_kind), int(device), int(bucket_bits), int(flags),
                            C.c_void_p(stream) if stream else None)
        rc = self._lib.grmkm_create(C.byref(cfg), C.byref(self._ctx))
        if rc != native.OK:
            msg = self._lib.grmkm_last_error(None)
            raise GrmkmError(rc, msg.decode() if msg else "grmkm_create failed")

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx:
            self._lib.grmkm_destroy(self._ctx)
            self._ctx = C.c_void_p()
        self._keep = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != native.OK:
            msg = self._lib.grmkm_last_error(self._ctx)
            raise GrmkmError(rc, msg.decode() if msg else "")

    # -- inputs -----------------------------------------------------------------------------
    def reset(self):
        self._check(self._lib.grmkm_reset(self._ctx))
        self._keep = []
        self._rows = self._declared = 0

    def add_genome_bytes(self, row: int, data) -> None:
        """data: bytes / bytearray / memoryview / uint8 ndarray (borrowed until build returns)."""
        if isinstance(data, np.ndarray):
            arr = np.ascontiguousarray(data, dtype=np.uint8)
        else:
            arr = np.frombuffer(data, dtype=np.uint8)
        self._keep.append(arr)
        self._check(self._lib.grmkm_add_genome_bytes(self._ctx, int(row), C.c_void_p(arr.ctypes.data), arr.size))
        self._rows = max(self._rows, int(row) + 1)

    def add_genome_device(self, row: int, dev_ptr: int, n_bytes: int) -> None:
        self._check(self._lib.grmkm_add_genome_device(self._ctx, int(row), C.c_void_p(int(dev_ptr)), int(n_bytes)))
        self._rows = max(self._rows, int(row) + 1)

    def add_genomes(self, rows, data, lens=None, on_device: bool = False) -> None:
        """Every input of the build in one call.  rows[i] = genome row of input i; data = device pointers (ints,
        with lens) when on_device, else host buffers (bytes / uint8 arrays, borrowed until build returns)."""
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        if on_device:
            ptrs = np.ascontiguousarray(data, dtype=np.uint64)
            lens = np.ascontiguousarray(lens, dtype=np.uint64)
        else:
            arrs = [np.ascontiguousarray(d, dtype=np.uint8) if isinstance(d, np.ndarray) else np.frombuffer(d, dtype=np.uint8)
                    for d in data]
            self._keep.extend(arrs)
            ptrs = np.array([a.ctypes.data for a in arrs], dtype=np.uint64)
            lens = np.array([a.size for a in arrs], dtype=np.uint64)
        if not (len(rows) == len(ptrs) == len(lens)):
            raise ValueError("rows, data and lens differ in length")
        self._check(self._lib.grmkm_add_genomes(self._ctx, len(rows), C.c_void_p(rows.ctypes.data), C.c_void_p(ptrs.ctypes.data),
                                                C.c_void_p(lens.ctypes.data), int(bool(on_device))))
        if len(rows):
            self._rows = max(self._rows, int(rows.max()) + 1)

    def add_genome_files(self, row: int, paths: Sequence[str]) -> None:
        paths = [paths] if isinstance(paths, (str, bytes)) else list(paths)
        arr = (C.c_char_p * max(len(paths), 1))(*[p.encode() if isinstance(p, str) else p for p in paths])
        self._check(self._lib.grmkm_add_genome_files(self._ctx, int(row), arr, len(paths)))
        self._rows = max(self._rows, int(row) + 1)

    def set_genome_count(self, n: int) -> None:
        self._check(self._lib.grmkm_set_genome_count(self._ctx, int(n)))
        self._declared = int(n)

    # -- build + results ----------------------------------------------------------------------
    def build(self) -> "KmerMatrixBuilder":
        self._check(self._lib.grmkm_build(self._ctx))
        return self

    @property
    def dims(self) -> tuple[int, int, int]:
        u, w, g = C.c_uint64(), C.c_uint32(), C.c_uint32()
        self._check(self._lib.grmkm_dims(self._ctx, C.byref(u), C.byref(w), C.byref(g)))
        return int(u.value), int(w.value), int(g.value)

    @property
    def stats(self) -> dict:
        s = native.Stats()
        self._check(self._lib.grmkm_get_stats(self._ctx, C.byref(s)))
        return s.asdict()

    @property
    def times(self) -> dict:
        t = native.Times()
        self._check(self._lib.grmkm_stage_times(self._ctx, C.byref(t)))
        return t.asdict()

    def kmers(self) -> np.ndarray:
        U, _, _ = self.dims
        out = np.empty(U, dtype=np.uint64)
        self._check(self._lib.grmkm_copy_kmers_packed(self._ctx, C.c_void_p(out.ctypes.data), U))
        return out

    def matrix(self) -> np.ndarray:
        U, W, _ = self.dims
        out = np.empty((W, U), dtype=np.uint64)
        self._check(self._lib.grmkm_copy_matrix(self._ctx, C.c_void_p(out.ctypes.data), U * W))
        return out

    def columns(self, idx) -> np.ndarray:
        """The (ceil(G/64) x len(idx)) words of columns ``idx``, packed on the device (grmkm_copy_columns): a few columns
        without copying the whole matrix."""
        _, W, _ = self.dims
        idx = np.ascontiguousarray(np.asarray(idx, dtype=np.uint64).reshape(-1))
        out = np.empty((W, idx.size), dtype=np.uint64)
        self._check(self._lib.grmkm_copy_columns(self._ctx, C.c_void_p(idx.ctypes.data), idx.size,
                                                 C.c_void_p(out.ctypes.data), out.size))
        return out

    def result_host(self) -> tuple[np.ndarray, np.ndarray]:
        """(kmers[U], matrix[W][U]) as views of the context's page-locked result buffer: one device->host
        copy at PCIe speed.  The views are valid until the next build / reset / close; copy them to keep them."""
        U, W, _ = self.dims
        a, b = C.c_void_p(), C.c_void_p()
        self._check(self._lib.grmkm_host_result(self._ctx, C.byref(a), C.byref(b)))
        if U == 0:
            return np.empty(0, dtype=np.uint64), np.empty((W, 0), dtype=np.uint64)
        km = np.ctypeslib.as_array(C.cast(a, C.POINTER(C.c_uint64)), shape=(U,))
        mat = np.ctypeslib.as_array(C.cast(b, C.POINTER(C.c_uint64)), shape=(W, U))
        return km, mat

    def kmer_strings(self) -> np.ndarray:
        U, _, _ = self.dims
        out = np.empty(U, dtype=f"S{self.k}")
        self._check(self._lib.grmkm_copy_kmer_strings(self._ctx, C.c_void_p(out.ctypes.data), U * self.k))
        return out

    def tsv(self, names: Iterable[str]) -> np.ndarray:
        """Ray Surveyor style KmerMatrix.tsv as a uint8 array (write with .tofile)."""
        names = [n.encode() if isinstance(n, str) else n for n in names]
        U, _, G = self.dims
        if len(names) != G:
            raise ValueError(f"{len(names)} names for {G} genomes")
        arr = (C.c_char_p * max(G, 1))(*names)
        need = C.c_uint64()
        rc = self._lib.grmkm_format_tsv(self._ctx, arr, None, 0, C.byref(need))
        if rc not in (native.OK, native.E_CAPACITY):
            self._check(rc)
        out = np.empty(int(need.value), dtype=np.uint8)
        self._check(self._lib.grmkm_format_tsv(self._ctx, arr, C.c_void_p(out.ctypes.data), out.size, C.byref(need)))
        return out

    # -- kernels over the resident result ------------------------------------------------------
    def checksum(self) -> tuple[int, int]:
        """Order-independent 128-bit digest of the columns (two wrapping 64-bit sums); the digests of the ranks'
        slices of a multi-GPU build add up to the digest of the one-GPU matrix (bench.py parity_check)."""
        out = (C.c_uint64 * 2)()
        self._check(self._lib.grmkm_result_checksum(self._ctx, out))
        return int(out[0]), int(out[1])

    def sum_rows(self, row_mask) -> np.ndarray:
        """Per column, the number of masked genome rows that hold the k-mer: popcount(matrix[:, j] & row_mask)
        summed over the word rows (rules.py:201-267).  row_mask: uint64[W], genome g at bit 63-(g%64) of word g//64."""
        U, W, _ = self.dims
        mask = np.ascontiguousarray(row_mask, dtype=np.uint64)
        if mask.shape != (W,):
            raise ValueError(f"row mask of {mask.shape} words for {W} matrix word rows")
        out = np.empty(U, dtype=np.uint32)
        self._check(self._lib.grmkm_sum_rows(self._ctx, C.c_void_p(mask.ctypes.data), W, C.c_void_p(out.ctypes.data), U))
        return out

    def gram(self) -> np.ndarray:
        """G x G shared-column counts (Ray Surveyor's similarity matrix)."""
        _, _, G = self.dims
        out = np.zeros((G, G), dtype=np.uint64)
        self._check(self._lib.grmkm_gram(self._ctx, C.c_void_p(out.ctypes.data), G * G))
        return out

    def tsv_pack(self, body: np.ndarray, row_width: int, k: int, n_tsv_cols: int, sel) -> np.ndarray:
        """from_tsv's bit packer: fixed-width TSV rows (uint8 body) -> matrix words [ceil(G/64)][n_rows]; matrix row g
        takes TSV column sel[g] (create.py:241-271, utils.py:133-156)."""
        body = np.ascontiguousarray(body, dtype=np.uint8).reshape(-1)
        sel = np.ascontiguousarray(sel, dtype=np.uint32)
        if row_width <= 0 or body.size % row_width:
            raise ValueError("the TSV body is not a whole number of rows")
        n_rows, G = body.size // row_width, int(sel.size)
        out = np.zeros(((G + 63) // 64, n_rows), dtype=np.uint64)
        self._check(self._lib.grmkm_tsv_pack(self._ctx, C.c_void_p(body.ctypes.data), n_rows, int(row_width), int(k),
                                             int(n_tsv_cols), G, C.c_void_p(sel.ctypes.data),
                                             C.c_void_p(out.ctypes.data), out.size))
        return out

    def load_result(self, kmers, matrix, n_genomes: int) -> "KmerMatrixBuilder":
        """An existing matrix (e.g. a .kover file's kmer_matrix, row-major ceil(G/64) x U words, and its packed k-mers)
        as this context's result, as if it had been built: every result-side call then works on it."""
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64).reshape(-1)
        matrix = np.ascontiguousarray(matrix, dtype=np.uint64)
        W = (int(n_genomes) + 63) // 64
        if matrix.shape != (W, kmers.size):
            raise ValueError(f"matrix of shape {matrix.shape} for {kmers.size} k-mers and {n_genomes} genomes")
        self._check(self._lib.grmkm_load_result(self._ctx, C.c_void_p(kmers.ctypes.data), C.c_void_p(matrix.ctypes.data),
                                                kmers.size, int(n_genomes)))
        return self

    def patterns(self, dst: "KmerMatrixBuilder", column_class=None, with_stats: bool = False):
        """The distinct presence patterns of this result (grmkm_patterns): columns with equal words (and equal
        ``column_class`` byte, 0..3, when given) form one pattern, patterns numbered by their first column.  ``dst``
        (another builder on this device) receives the P x W pattern matrix, the k-mers of the patterns' first columns
        and their multiplicities.  -> (pattern_of_column uint32[U], members uint32[U], member_offsets uint64[P + 1]):
        the members of pattern p, ascending, are members[member_offsets[p]:member_offsets[p + 1]].  with_stats: also
        the call's statistics (rounds, P, device ms) as a dict."""
        U, _, _ = self.dims
        cls = None
        if column_class is not None:
            cls = np.ascontiguousarray(column_class)
            if cls.shape != (U,) or cls.dtype.kind not in "biu" or (U and (cls.min() < 0 or cls.max() > 255)):
                raise ValueError(f"column_class must hold one integer class per column ({U}), not {cls.shape} {cls.dtype}")
            cls = cls.astype(np.uint8)
        pattern_of = np.empty(U, dtype=np.uint32)
        members = np.empty(U, dtype=np.uint32)
        offsets = np.empty(U + 1, dtype=np.uint64)
        st = native.PatternStats()
        st.struct_size = C.sizeof(native.PatternStats)
        self._check(self._lib.grmkm_patterns(self._ctx, None if cls is None else C.c_void_p(cls.ctypes.data), dst._ctx,
                                             C.c_void_p(pattern_of.ctypes.data), U, C.c_void_p(members.ctypes.data), U,
                                             C.c_void_p(offsets.ctypes.data), U + 1, C.byref(st)))
        out = (pattern_of, members, offsets[: int(st.n_patterns) + 1].copy())
        return (*out, st.asdict()) if with_stats else out

    def _sharded(self, fn: str, shard, *args):
        """Call grmkm_<fn> (shard None), or grmkm_<fn>_sharded on this context's slice of the columns.  shard: rank,
        world, col_offset, n_kmers_total and exchange, whose allgather(bytes) returns every rank's bytes in rank order
        (learning.ShardedRuleClassifications).  The ctypes callback and the last received bytes live until the call
        returns."""
        if shard is None:
            return self._check(getattr(self._lib, "grmkm_" + fn)(self._ctx, *args))
        keep = {}

        def exchange(user, send, n, recv, sizes):
            try:
                blocks = shard.exchange.allgather(C.string_at(send, n) if n else b"")
                if len(blocks) != shard.world:
                    raise RuntimeError(f"the exchange returned {len(blocks)} blocks for {shard.world} ranks")
                keep["recv"] = C.create_string_buffer(b"".join(blocks), max(1, sum(map(len, blocks))))
                recv[0] = C.cast(keep["recv"], C.c_void_p)
                for r, b in enumerate(blocks):
                    sizes[r] = len(b)
                return 0
            except BaseException as e:          # an exception must not cross the C frames
                keep["error"] = e
                return 1

        cb = native.EXCHANGE_FN(exchange)
        sh = native.Shard(C.sizeof(native.Shard), int(shard.rank), int(shard.world), 0, int(shard.col_offset),
                          int(shard.n_kmers_total), cb, None)
        rc = getattr(self._lib, "grmkm_" + fn + "_sharded")(self._ctx, *args, C.byref(sh))
        if rc != native.OK and "error" in keep:
            msg = self._lib.grmkm_last_error(self._ctx)
            raise GrmkmError(rc, msg.decode() if msg else "") from keep["error"]
        self._check(rc)

    def scm_run(self, jobs, blacklist=(), shard=None) -> list[tuple[np.ndarray, np.ndarray]]:
        """Set Covering Machine fits on the resident matrix, all in one grmkm_scm_run.  jobs: (model_type, p, max_rules,
        tiebreak, pos_mask, neg_mask) with masks of ceil(G/64) uint64 words.  -> per fit (steps, equivalent rules):
        steps is a structured array with the fields of grmkm_scm_step.  shard: this context holds one slice of the
        columns (see _sharded); every rank gets the global result, rule indices global."""
        _, W, _ = self.dims
        masks, arr = [], (native.ScmJob * max(1, len(jobs)))()
        for i, (model_type, p, max_rules, tiebreak, pos, neg) in enumerate(jobs):
            pos = np.ascontiguousarray(pos, dtype=np.uint64)
            neg = np.ascontiguousarray(neg, dtype=np.uint64)
            if pos.shape != (W,) or neg.shape != (W,):
                raise ValueError(f"example masks of {pos.shape} / {neg.shape} words for {W} matrix word rows")
            masks += [pos, neg]
            arr[i] = native.ScmJob(C.sizeof(native.ScmJob), int(model_type), int(max_rules), int(bool(tiebreak)), float(p),
                                   pos.ctypes.data, neg.ctypes.data)
        bl = np.ascontiguousarray(blacklist if blacklist is not None else (), dtype=np.uint64).reshape(-1)
        self._sharded("scm_run", shard, len(jobs), arr, C.c_void_p(bl.ctypes.data), bl.size)
        out = []
        step_dtype = np.dtype([("rule", np.uint64), ("utility", np.float64), ("positive_errors", np.uint32),
                               ("negative_covers", np.uint32), ("equiv_offset", np.uint64), ("equiv_count", np.uint64)])
        for f in range(len(jobs)):
            ns, ne = C.c_uint64(), C.c_uint64()
            rc = self._lib.grmkm_scm_result(self._ctx, f, None, 0, C.byref(ns), None, 0, C.byref(ne))
            if rc not in (native.OK, native.E_CAPACITY):
                self._check(rc)
            steps = np.zeros(ns.value, dtype=step_dtype)
            eq = np.zeros(ne.value, dtype=np.uint64)
            self._check(self._lib.grmkm_scm_result(self._ctx, f, C.c_void_p(steps.ctypes.data), steps.size, C.byref(ns),
                                                   C.c_void_p(eq.ctypes.data), eq.size, C.byref(ne)))
            out.append((steps, eq))
        return out

    CART_NODE_DTYPE = np.dtype([("rule", np.uint64), ("score", np.float64), ("depth", np.uint32), ("n_pos", np.uint32),
                                ("n_neg", np.uint32), ("present_child", np.uint32), ("absent_child", np.uint32),
                                ("prediction", np.uint32), ("equiv_offset", np.uint64), ("equiv_count", np.uint64),
                                ("equiv_total", np.uint64)])

    def cart_run(self, jobs, blacklist=(), shard=None) -> list[tuple[np.ndarray, np.ndarray]]:
        """CART trees on the resident matrix, all in one grmkm_cart_run.  jobs: (max_depth, min_samples_split,
        equiv_cap, w_neg, w_pos, pos_mask, neg_mask) with masks of ceil(G/64) uint64 words.  -> per tree (nodes,
        equivalent rules): nodes is a structured array with the fields of grmkm_cart_node, in breadth-first order.
        shard: as for scm_run."""
        _, W, _ = self.dims
        masks, arr = [], (native.CartJob * max(1, len(jobs)))()
        for i, (max_depth, min_samples_split, equiv_cap, w_neg, w_pos, pos, neg) in enumerate(jobs):
            pos = np.ascontiguousarray(pos, dtype=np.uint64)
            neg = np.ascontiguousarray(neg, dtype=np.uint64)
            if pos.shape != (W,) or neg.shape != (W,):
                raise ValueError(f"example masks of {pos.shape} / {neg.shape} words for {W} matrix word rows")
            masks += [pos, neg]
            arr[i] = native.CartJob(C.sizeof(native.CartJob), int(max_depth), int(min_samples_split), 0, int(equiv_cap),
                                    float(w_neg), float(w_pos), pos.ctypes.data, neg.ctypes.data)
        bl = np.ascontiguousarray(blacklist if blacklist is not None else (), dtype=np.uint64).reshape(-1)
        self._sharded("cart_run", shard, len(jobs), arr, C.c_void_p(bl.ctypes.data), bl.size)
        out = []
        for t in range(len(jobs)):
            nn, ne = C.c_uint64(), C.c_uint64()
            rc = self._lib.grmkm_cart_result(self._ctx, t, None, 0, C.byref(nn), None, 0, C.byref(ne))
            if rc not in (native.OK, native.E_CAPACITY):
                self._check(rc)
            nodes = np.zeros(nn.value, dtype=self.CART_NODE_DTYPE)
            eq = np.zeros(ne.value, dtype=np.uint64)
            self._check(self._lib.grmkm_cart_result(self._ctx, t, C.c_void_p(nodes.ctypes.data), nodes.size, C.byref(nn),
                                                    C.c_void_p(eq.ctypes.data), eq.size, C.byref(ne)))
            out.append((nodes, eq))
        return out

    EVAL_NODE_DTYPE = np.dtype([("kmer", np.uint64), ("present_child", np.uint32), ("absent_child", np.uint32)])

    def eval_run(self, jobs, shard=None) -> list[np.ndarray]:
        """Fitted models scored on example sets of the resident matrix, all in one grmkm_eval_run (one launch, one copy
        of the counts).  jobs: (kind, model_type, items, pos_mask, neg_mask) with masks of ceil(G/64) uint64 words.
        kind native.EVAL_SCM: items = the model's rule indices (< 2U), model_type native.SCM_CONJUNCTION / _DISJUNCTION
        -> (R + 1, 2) counts (fn, fp) of the prefixes of 0..R rules.  kind native.EVAL_CART: model_type 0, items = nodes
        with the fields of EVAL_NODE_DTYPE (kmer UINT64_MAX: leaf) -> (n, 2) counts (pos, neg) of the examples reaching
        each node.  shard: as for scm_run (rule and k-mer indices global)."""
        _, W, _ = self.dims
        keep, arr, sizes = [], (native.EvalJob * max(1, len(jobs)))(), []
        for i, (kind, model_type, items, pos, neg) in enumerate(jobs):
            pos = np.ascontiguousarray(pos, dtype=np.uint64)
            neg = np.ascontiguousarray(neg, dtype=np.uint64)
            if pos.shape != (W,) or neg.shape != (W,):
                raise ValueError(f"example masks of {pos.shape} / {neg.shape} words for {W} matrix word rows")
            if kind == native.EVAL_SCM:
                items = np.ascontiguousarray(np.asarray(items, dtype=np.uint64).reshape(-1))
                rules, nodes, pairs = items.ctypes.data, None, items.size + 1
            else:
                items = np.ascontiguousarray(items, dtype=self.EVAL_NODE_DTYPE).reshape(-1)
                rules, nodes, pairs = None, items.ctypes.data, items.size
            keep += [pos, neg, items]
            sizes.append(pairs)
            arr[i] = native.EvalJob(C.sizeof(native.EvalJob), int(kind), int(model_type), 0, items.size, rules, nodes,
                                    pos.ctypes.data, neg.ctypes.data)
        counts = np.zeros((sum(sizes), 2), dtype=np.uint32)
        self._sharded("eval_run", shard, len(jobs), arr, C.c_void_p(counts.ctypes.data), counts.size)
        return np.split(counts, np.cumsum(sizes)[:-1]) if sizes else []

    @property
    def query_genome_count(self) -> int:
        """G of a build of the inputs added since the last reset: max row + 1, or set_genome_count when larger."""
        return max(self._rows, self._declared)

    def query(self, kmers, with_stats: bool = False):
        """Which genome rows of the inputs added since the last reset hold which k-mers, without a build: uint64
        (ceil(G/64), len(kmers)), genome g at bit 63 - g % 64 of word row g // 64 (the matrix's layout).  kmers: packed
        as ``kmers()`` returns them, either strand, duplicates allowed; column i is about the canonical form of
        kmers[i], set for a genome whose windows hold it at least min_abundance times.  The resident result, stats and
        fits are left as they are.  with_stats: also return the call's statistics as a dict."""
        q = np.ascontiguousarray(np.asarray(kmers, dtype=np.uint64).reshape(-1))
        G = self.query_genome_count
        out = np.zeros(((G + 63) // 64, q.size), dtype=np.uint64)
        st = native.QueryStats()
        st.struct_size = C.sizeof(native.QueryStats)
        self._check(self._lib.grmkm_query(self._ctx, C.c_void_p(q.ctypes.data), q.size, C.c_void_p(out.ctypes.data),
                                          out.size, C.byref(st)))
        return (out, st.asdict()) if with_stats else out

    def device_result(self) -> tuple[int, int, int]:
        """(device pointer of kmers[U], device pointer of the matrix, row pitch in words): word row w of the matrix
        starts at pointer + 8 * w * pitch."""
        a, b, p = C.c_void_p(), C.c_void_p(), C.c_uint64()
        self._check(self._lib.grmkm_device_result(self._ctx, C.byref(a), C.byref(b), C.byref(p)))
        return int(a.value or 0), int(b.value or 0), int(p.value)


class BuildPipeline:
    """Several builds in flight on ONE GPU (a series of datasets: one per antibiotic / species / parameter set).

    ``depth`` contexts, each with its own stream, staging halves, page-locked result buffer and worker thread.
    Build i + 1's text crosses PCIe host->device while build i's dedupe / expand / aggregate kernels and its
    device->host copy of (kmers, matrix) are still in flight: the two directions of the link and the SMs are all
    busy at once, so a stream of builds runs at the speed of the slowest leg (the H2D copy) instead of the sum of
    the legs.  Every build still copies all of its own input in and all of its own result out.

    submit(rows, data[, n_genomes]) -> Future of (kmers, matrix, stats): views of the slot's page-locked result buffer, valid
    until ``depth`` further submissions have been made (copy them to keep them longer).
    """

    def __init__(self, depth: int = 2, streams: Sequence[int] | None = None, **builder_kw):
        """streams: one CUDA stream handle per slot (default: every slot creates its own)."""
        import concurrent.futures as cf
        if depth < 1:
            raise ValueError("depth must be at least 1")
        if streams is not None and len(streams) != depth:
            raise ValueError("one stream per slot")
        builder_kw.pop("stream", None)
        self.slots = [KmerMatrixBuilder(stream=streams[i] if streams else None, **builder_kw) for i in range(depth)]
        self._workers = [cf.ThreadPoolExecutor(max_workers=1) for _ in range(depth)]
        self._n = 0

    @staticmethod
    def _run(b: KmerMatrixBuilder, rows, data, lens, on_device, n_genomes):
        # (the slot's previous build has finished: one worker per slot.  The library lets the H2D legs of builds in
        # different contexts of one device follow one another -- grmkm_api.cu, h2d gate -- so the builds fall into step:
        # one copies its text in while the other computes and copies its result out.)
        b.reset()
        if n_genomes:
            b.set_genome_count(n_genomes)
        b.add_genomes(rows, data, lens, on_device)
        b.build()
        km, mat = b.result_host()
        return km, mat, b.stats

    def submit(self, rows, data, lens=None, on_device: bool = False, n_genomes: int = 0):
        i = self._n
        self._n += 1
        s = i % len(self.slots)
        return self._workers[s].submit(self._run, self.slots[s], rows, data, lens, on_device, n_genomes)

    def close(self):
        for w in self._workers:
            w.shutdown(wait=True)
        for b in self.slots:
            b.close()
        self.slots = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def build_matrix(genomes: Sequence, k: int = 31, min_abundance: int = 1, keep_singletons: bool = False,
                 input_kind: int = FASTA, **kw):
    """One-shot helper: genomes = list (row order) of bytes or lists of bytes.  Returns (kmers, matrix, stats)."""
    with KmerMatrixBuilder(k=k, min_abundance=min_abundance, keep_singletons=keep_singletons,
                           input_kind=input_kind, **kw) as b:
        b.set_genome_count(len(genomes))
        for row, files in enumerate(genomes):
            if isinstance(files, (bytes, bytearray, memoryview, np.ndarray)):
                files = [files]
            for f in files:
                b.add_genome_bytes(row, f)
        b.build()
        return b.kmers(), b.matrix(), b.stats
