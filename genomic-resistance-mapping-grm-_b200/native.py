"""ctypes binding of libgrmkm.so (include/grmkm.h).  Fails loudly: no library or no GPU -> error."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GRMKM_LIB") or os.path.join(_HERE, "libgrmkm.so")   # GRMKM_LIB: another build of the same library (kernel experiments)
ABI_VERSION = 16

OK = 0
E_INVALID, E_UNSUPPORTED_K, E_NOMEM, E_CUDA, E_IO, E_CAPACITY, E_NO_DEVICE, E_UNSUPPORTED = -1, -2, -3, -4, -5, -6, -7, -8
FASTA, FASTQ = 0, 1
FLAG_COUNTS = 32      # pooled count table (dsk mode): matrix row 0 = abundance of the k-mer over all inputs

# every symbol include/grmkm.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "grmkm_abi_version", "grmkm_device_count", "grmkm_create", "grmkm_destroy", "grmkm_last_error", "grmkm_reset",
    "grmkm_add_genome_bytes", "grmkm_add_genome_device", "grmkm_add_genome_files", "grmkm_add_genomes", "grmkm_set_genome_count",
    "grmkm_build", "grmkm_dims", "grmkm_get_stats", "grmkm_stage_times", "grmkm_copy_kmers_packed",
    "grmkm_copy_kmer_strings", "grmkm_copy_matrix", "grmkm_format_tsv", "grmkm_device_result", "grmkm_host_result",
    "grmkm_synth_fasta_device", "grmkm_build_partial", "grmkm_export_partials", "grmkm_export_partials_peers", "grmkm_merge_partials",
    "grmkm_plan_bucket_bits", "grmkm_set_bucket_bits", "grmkm_set_exchange_rank",
    "grmkm_result_checksum", "grmkm_sum_rows", "grmkm_gram", "grmkm_tsv_pack",
    "grmkm_load_result", "grmkm_scm_run", "grmkm_scm_result",
    "grmkm_cart_run", "grmkm_cart_result", "grmkm_query", "grmkm_eval_run",
    "grmkm_scm_run_sharded", "grmkm_cart_run_sharded", "grmkm_eval_run_sharded", "grmkm_copy_columns",
    "grmkm_patterns",
]
SCM_CONJUNCTION, SCM_DISJUNCTION = 0, 1
EVAL_SCM, EVAL_CART = 0, 1


class GrmkmError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libgrmkm error {code}: {message}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("k", C.c_uint32), ("min_abundance", C.c_uint32),
                ("keep_singletons", C.c_uint32), ("input_kind", C.c_uint32), ("device", C.c_int32),
                ("bucket_bits", C.c_uint32), ("flags", C.c_uint32), ("stream", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("n_bases", C.c_uint64), ("n_windows", C.c_uint64), ("n_input_bytes", C.c_uint64),
                ("n_records", C.c_uint64), ("n_kmers", C.c_uint64), ("n_distinct", C.c_uint64),
                ("n_words", C.c_uint32), ("n_genomes", C.c_uint32), ("n_buckets", C.c_uint32),
                ("n_launches", C.c_uint32), ("h2d_bytes", C.c_uint64), ("device_bytes", C.c_uint64),
                ("n_splits", C.c_uint64), ("n_region_overflows", C.c_uint64), ("n_units", C.c_uint64),
                ("n_unit_entries", C.c_uint64), ("n_wide", C.c_uint64), ("n_unit_buckets", C.c_uint32),
                ("n_rounds", C.c_uint32), ("n_solid_records", C.c_uint64)]

    def asdict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


class Times(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("h2d", "parse", "pack", "count", "scatter", "abundance", "aggregate",
                                         "sort", "total", "bounds", "dedupe", "expand")]

    def asdict(self):
        return {n: float(getattr(self, n)) for n, _ in self._fields_}


class ScmJob(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("model_type", C.c_uint32), ("max_rules", C.c_uint32),
                ("tiebreak", C.c_uint32), ("p", C.c_double), ("pos", C.c_void_p), ("neg", C.c_void_p)]


class ScmStep(C.Structure):
    _fields_ = [("rule", C.c_uint64), ("utility", C.c_double), ("positive_errors", C.c_uint32),
                ("negative_covers", C.c_uint32), ("equiv_offset", C.c_uint64), ("equiv_count", C.c_uint64)]


class CartJob(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("max_depth", C.c_uint32), ("min_samples_split", C.c_uint32),
                ("reserved", C.c_uint32), ("equiv_cap", C.c_uint64), ("w_neg", C.c_double), ("w_pos", C.c_double),
                ("pos", C.c_void_p), ("neg", C.c_void_p)]


class CartNode(C.Structure):
    _fields_ = [("rule", C.c_uint64), ("score", C.c_double), ("depth", C.c_uint32), ("n_pos", C.c_uint32),
                ("n_neg", C.c_uint32), ("present_child", C.c_uint32), ("absent_child", C.c_uint32),
                ("prediction", C.c_uint32), ("equiv_offset", C.c_uint64), ("equiv_count", C.c_uint64),
                ("equiv_total", C.c_uint64)]


class QueryStats(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_jobs", C.c_uint32), ("n_queries", C.c_uint64),
                ("n_bases", C.c_uint64), ("n_windows", C.c_uint64), ("n_records", C.c_uint64),
                ("n_input_bytes", C.c_uint64), ("n_hits", C.c_uint64), ("ms", C.c_float)]

    def asdict(self):
        return {n: (float if n == "ms" else int)(getattr(self, n)) for n, _ in self._fields_ if n != "struct_size"}


class EvalNode(C.Structure):
    _fields_ = [("kmer", C.c_uint64), ("present_child", C.c_uint32), ("absent_child", C.c_uint32)]


class EvalJob(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("kind", C.c_uint32), ("model_type", C.c_uint32), ("reserved", C.c_uint32),
                ("n_items", C.c_uint64), ("rules", C.c_void_p), ("nodes", C.c_void_p), ("pos", C.c_void_p),
                ("neg", C.c_void_p)]


class PatternStats(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_rounds", C.c_uint32), ("n_patterns", C.c_uint64), ("ms", C.c_float)]

    def asdict(self):
        return {n: (float if n == "ms" else int)(getattr(self, n)) for n, _ in self._fields_ if n != "struct_size"}


# int exchange(void* user, const void* send, uint64_t n, const void** recv, uint64_t* sizes): the all-gather of the
# sharded runs
EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64))


class Shard(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("rank", C.c_uint32), ("n_ranks", C.c_uint32), ("reserved", C.c_uint32),
                ("col_offset", C.c_uint64), ("n_kmers_total", C.c_uint64), ("exchange", EXCHANGE_FN),
                ("user", C.c_void_p)]


_lib = None


def load() -> C.CDLL:
    """Load libgrmkm.so; raise if it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
                          "(there is no CPU fallback for the k-mer matrix path)")
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    sig = {
        "grmkm_abi_version": (i32, []),
        "grmkm_device_count": (i32, []),
        "grmkm_create": (i32, [C.POINTER(Config), C.POINTER(vp)]),
        "grmkm_destroy": (None, [vp]),
        "grmkm_last_error": (C.c_char_p, [vp]),
        "grmkm_reset": (i32, [vp]),
        "grmkm_add_genome_bytes": (i32, [vp, u32, vp, u64]),
        "grmkm_add_genome_device": (i32, [vp, u32, vp, u64]),
        "grmkm_add_genome_files": (i32, [vp, u32, C.POINTER(C.c_char_p), i32]),
        "grmkm_set_genome_count": (i32, [vp, u32]),
        "grmkm_build": (i32, [vp]),
        "grmkm_dims": (i32, [vp, C.POINTER(u64), C.POINTER(u32), C.POINTER(u32)]),
        "grmkm_get_stats": (i32, [vp, C.POINTER(Stats)]),
        "grmkm_stage_times": (i32, [vp, C.POINTER(Times)]),
        "grmkm_copy_kmers_packed": (i32, [vp, vp, u64]),
        "grmkm_copy_kmer_strings": (i32, [vp, vp, u64]),
        "grmkm_copy_matrix": (i32, [vp, vp, u64]),
        "grmkm_add_genomes": (i32, [vp, u32, vp, vp, vp, i32]),
        "grmkm_format_tsv": (i32, [vp, C.POINTER(C.c_char_p), vp, u64, C.POINTER(u64)]),
        "grmkm_device_result": (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64)]),
        "grmkm_host_result": (i32, [vp, C.POINTER(vp), C.POINTER(vp)]),
        "grmkm_synth_fasta_device": (i32, [vp, vp, u64, vp, u64]),
        "grmkm_build_partial": (i32, [vp, u32, C.POINTER(u64)]),
        "grmkm_export_partials": (i32, [vp, vp, u64]),
        "grmkm_export_partials_peers": (i32, [vp, u32, vp, vp]),
        "grmkm_merge_partials": (i32, [vp, vp, u32, u32, C.POINTER(u64), C.POINTER(u32), u32]),
        "grmkm_plan_bucket_bits": (i32, [vp, C.POINTER(u32)]),
        "grmkm_set_bucket_bits": (i32, [vp, u32]),
        "grmkm_set_exchange_rank": (i32, [vp, u32]),
        "grmkm_result_checksum": (i32, [vp, C.POINTER(u64)]),
        "grmkm_sum_rows": (i32, [vp, vp, u32, vp, u64]),
        "grmkm_gram": (i32, [vp, vp, u64]),
        "grmkm_tsv_pack": (i32, [vp, vp, u64, u32, u32, u32, u32, vp, vp, u64]),
        "grmkm_load_result": (i32, [vp, vp, vp, u64, u32]),
        "grmkm_scm_run": (i32, [vp, u32, vp, vp, u64]),
        "grmkm_scm_result": (i32, [vp, u32, vp, u64, C.POINTER(u64), vp, u64, C.POINTER(u64)]),
        "grmkm_cart_run": (i32, [vp, u32, vp, vp, u64]),
        "grmkm_cart_result": (i32, [vp, u32, vp, u64, C.POINTER(u64), vp, u64, C.POINTER(u64)]),
        "grmkm_query": (i32, [vp, vp, u64, vp, u64, C.POINTER(QueryStats)]),
        "grmkm_eval_run": (i32, [vp, u32, vp, vp, u64]),
        "grmkm_scm_run_sharded": (i32, [vp, u32, vp, vp, u64, C.POINTER(Shard)]),
        "grmkm_cart_run_sharded": (i32, [vp, u32, vp, vp, u64, C.POINTER(Shard)]),
        "grmkm_eval_run_sharded": (i32, [vp, u32, vp, vp, u64, C.POINTER(Shard)]),
        "grmkm_copy_columns": (i32, [vp, vp, u64, vp, u64]),
        "grmkm_patterns": (i32, [vp, vp, vp, vp, u64, vp, u64, vp, u64, C.POINTER(PatternStats)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.grmkm_abi_version() != ABI_VERSION:
        raise ImportError(f"libgrmkm ABI {L.grmkm_abi_version()} != expected {ABI_VERSION}; rebuild")
    _lib = L
    return L
