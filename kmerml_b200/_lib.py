"""ctypes binding of libkmerml_b200.so (include/kmerml_b200.h).

The product path fails loudly when the CUDA library is missing or no B200 is
present: there is no CPU fallback anywhere in this package.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("KMERML_LIB") or os.path.join(_HERE, "libkmerml_b200.so")    # KMERML_LIB: A/B builds

OK = 0
FLAG_CANONICAL = 1
FLAG_NO_PARTITION = 2
FLAG_FREQ_ON_DEVICE = 4
FLAG_K8_AS_9 = 8
FLAG_WIDE_D2H = 16
FLAG_NO_NIBBLES = 32
MAX_DENSE_K = 14
MAX_K = 32
SKETCH_MAX = 16384
SKETCH_METRIC_MASH = 0
SKETCH_METRIC_JACCARD = 1

_lib = None


class Profile(ctypes.Structure):
    _fields_ = [("launches", ctypes.c_uint64), ("count_launches", ctypes.c_uint64),
                ("ms_count", ctypes.c_double), ("ms_cascade", ctypes.c_double),
                ("ms_finalize", ctypes.c_double), ("ms_other", ctypes.c_double),
                ("ms_partition", ctypes.c_double), ("ms_bucket", ctypes.c_double)]


class KmermlError(RuntimeError):
    pass


def load():
    """Load the shared library (no GPU needed for loading, only for calling)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m kmerml_b200.build` "
            "(nvcc, sm_100a). kmerml_b200 has no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, u32, u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint, ctypes.c_uint64
    L.kmerml_version.restype = i32
    L.kmerml_last_error.restype = ctypes.c_char_p
    L.kmerml_ctx_create.argtypes = [i32, ctypes.POINTER(vp)]
    L.kmerml_ctx_destroy.argtypes = [vp]
    L.kmerml_ctx_sm_count.argtypes = [vp]
    L.kmerml_ctx_set_host_threads.argtypes = [vp, i32]
    L.kmerml_row_len.restype = u64
    L.kmerml_row_len.argtypes = [vp, i32]
    p64 = ctypes.POINTER(ctypes.c_uint64)
    L.kmerml_count_dense_batch.argtypes = [vp, vp, vp, i32, vp, i32, i32, u32, vp, u64, vp, u64, vp, vp]
    L.kmerml_count_dense_host.argtypes = [vp, vp, vp, i32, vp, i32, i32, u32, vp, u64, vp, u64, vp]
    L.kmerml_compact_row_bytes.restype = u64
    L.kmerml_compact_row_bytes.argtypes = [vp, i32]
    L.kmerml_count_dense_host_compact.argtypes = [vp, vp, vp, i32, vp, i32, i32, u32, vp, u64, vp, u64, vp]
    L.kmerml_compact_expand.argtypes = [vp, i32, vp, i32, vp]
    L.kmerml_compact_row_overflowed.argtypes = [vp, i32, vp]
    L.kmerml_compact_row_used_bytes.restype = u64
    L.kmerml_compact_row_used_bytes.argtypes = [vp, i32, vp]
    L.kmerml_count_dense_range.argtypes = [vp, vp, u64, u64, u64, vp, i32, i32, u32, vp, vp, vp]
    L.kmerml_count_sparse.argtypes = [vp, vp, u64, i32, i32, u32, vp, vp, vp, u64, ctypes.POINTER(ctypes.c_uint64),
                                      ctypes.POINTER(ctypes.c_uint64), vp]
    L.kmerml_count_sparse_range.argtypes = [vp, vp, u64, u64, u64, i32, i32, u32, vp, vp, vp, u64,
                                            ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_uint64), vp]
    L.kmerml_emit_sparse_range.argtypes = [vp, vp, u64, u64, u64, i32, i32, u32, i32, vp, vp, u64, p64, vp, vp]
    L.kmerml_reduce_sparse_windows.argtypes = [vp, i32, vp, vp, u64, vp, vp, vp, u64, p64, vp]
    L.kmerml_sparse_fetch.argtypes = [vp, vp, vp, vp, u64, vp]
    L.kmerml_merge_sparse.argtypes = [vp, i32, vp, vp, vp, u64, vp, vp, vp, u64, ctypes.POINTER(ctypes.c_uint64), vp]
    L.kmerml_first_occurrence.argtypes = [vp, vp, u64, i32, i32, vp, vp]
    L.kmerml_find_records.argtypes = [vp, vp, u64, vp, u32, ctypes.POINTER(ctypes.c_uint32), vp]
    L.kmerml_records_short.argtypes = [vp, vp, u64, vp, u32, i32, vp, vp]
    L.kmerml_genome_stats.argtypes = [vp, vp, u64, vp, vp]
    L.kmerml_encode.argtypes = [vp, vp, u64, vp, vp, vp]
    L.kmerml_allreduce_counts.argtypes = [vp, vp, vp, u64, i32, i32, vp]
    L.kmerml_format_kmer_file.argtypes = [vp, i32, vp, vp, u32, u64, vp, u64, p64, p64, vp]
    L.kmerml_format_kmer_lines.argtypes = [vp, i32, vp, vp, u64, vp, u64, p64, vp]
    L.kmerml_parse_kmer_lines.argtypes = [vp, vp, vp, u64, vp, vp, ctypes.POINTER(ctypes.c_uint32), vp]
    L.kmerml_feature_keys.argtypes = [vp, vp, u64, vp, vp]
    L.kmerml_feature_line_lengths.argtypes = [vp, vp, vp, vp, vp, u64, vp, vp]
    L.kmerml_feature_write_lines.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, u64, vp, vp]
    L.kmerml_count_stats.argtypes = [vp, vp, u64, vp, vp]
    L.kmerml_column_stats.argtypes = [vp, vp, i32, u64, i32, u64, vp, vp, vp, vp]
    L.kmerml_static_features.argtypes = [vp, i32, i32, vp, vp]
    L.kmerml_normalize_rows.argtypes = [vp, vp, u64, vp, i32, u64, vp, u64, vp]
    L.kmerml_pairwise_distance.argtypes = [vp, vp, i32, u64, i32, u64, i32, vp, vp, vp]
    L.kmerml_pairwise_distance_rows.argtypes = [vp, vp, u64, i32, u64, i32, i32, i32, vp, vp, vp]
    L.kmerml_count_planes.argtypes = [vp, vp, u64, i32, u64, vp, u64, vp, vp, vp]
    L.kmerml_distance_rows_planes.argtypes = [vp, vp, u64, i32, i32, u64, vp, i32, i32, i32, vp, vp, vp]
    L.kmerml_sketch_batch.argtypes = [vp, vp, vp, i32, i32, i32, u32, i32, u64, vp, u64, vp, vp]
    L.kmerml_sketch_distance_rows.argtypes = [vp, vp, u64, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp]
    L.kmerml_profile_enable.argtypes = [vp, i32]
    L.kmerml_profile_read.argtypes = [vp, ctypes.POINTER(Profile), i32]
    for name in EXPORTS:
        fn = getattr(L, name)          # AttributeError here = header/library mismatch
        if fn.restype is ctypes.c_int and name not in ("kmerml_version", "kmerml_ctx_sm_count"):
            pass
    _lib = L
    return L


# every symbol include/kmerml_b200.h declares (checked by tests/test_cabi.py)
EXPORTS = [
    "kmerml_version", "kmerml_last_error", "kmerml_ctx_create", "kmerml_ctx_destroy",
    "kmerml_ctx_sm_count", "kmerml_row_len", "kmerml_count_dense_batch",
    "kmerml_count_dense_host", "kmerml_first_occurrence", "kmerml_profile_enable",
    "kmerml_profile_read", "kmerml_find_records", "kmerml_records_short", "kmerml_static_features",
    "kmerml_normalize_rows", "kmerml_pairwise_distance", "kmerml_count_dense_range",
    "kmerml_count_sparse", "kmerml_genome_stats", "kmerml_encode", "kmerml_allreduce_counts", "kmerml_format_kmer_file", "kmerml_format_kmer_lines",
    "kmerml_count_sparse_range", "kmerml_merge_sparse", "kmerml_pairwise_distance_rows", "kmerml_count_planes", "kmerml_distance_rows_planes", "kmerml_sparse_fetch", "kmerml_ctx_set_host_threads", "kmerml_count_stats", "kmerml_column_stats",
    "kmerml_compact_row_bytes", "kmerml_count_dense_host_compact", "kmerml_compact_expand", "kmerml_compact_row_overflowed", "kmerml_compact_row_used_bytes",
    "kmerml_parse_kmer_lines", "kmerml_feature_keys", "kmerml_feature_line_lengths", "kmerml_feature_write_lines",
    "kmerml_emit_sparse_range", "kmerml_reduce_sparse_windows",
    "kmerml_sketch_batch", "kmerml_sketch_distance_rows",
]


def check(status):
    if status != OK:
        msg = load().kmerml_last_error()
        raise KmermlError(f"kmerml_b200 error {status}: {msg.decode() if msg else '?'}")


class Context:
    """One per GPU (per host thread).  Wraps kmerml_ctx_create/destroy."""

    def __init__(self, device=0):
        self._lib = load()
        self._h = ctypes.c_void_p()
        check(self._lib.kmerml_ctx_create(int(device), ctypes.byref(self._h)))
        self.device = int(device)

    @property
    def handle(self):
        if not self._h:
            raise KmermlError("context already destroyed")
        return self._h

    @property
    def sm_count(self):
        return self._lib.kmerml_ctx_sm_count(self.handle)

    def set_host_threads(self, n):
        """Host threads that widen the narrow D2H format of count_dense_host (default: half the cores, <= 16)."""
        check(self._lib.kmerml_ctx_set_host_threads(self.handle, int(n)))

    def profile_enable(self, on=True):
        check(self._lib.kmerml_profile_enable(self.handle, 1 if on else 0))

    def profile_read(self, reset=True):
        p = Profile()
        check(self._lib.kmerml_profile_read(self.handle, ctypes.byref(p), 1 if reset else 0))
        return {f: getattr(p, f) for f, _ in Profile._fields_}

    def close(self):
        if self._h:
            self._lib.kmerml_ctx_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_contexts = {}


def context(device=0):
    """Context cache: one per (device, host thread), as include/kmerml_b200.h asks (a context's workspaces are
    not shared between threads)."""
    import threading
    key = (device, threading.get_ident())
    ctx = _contexts.get(key)
    if ctx is None:
        ctx = _contexts[key] = Context(device)
    return ctx
