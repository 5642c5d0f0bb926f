"""ctypes binding of include/pixelbox_b200.h.

There is no fallback of any kind: if the shared library has not been built this module raises,
and every compute entry point fails with PBX_E_NO_DEVICE when no sm_100 GPU is present.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("PBX_SO", os.path.join(HERE, "lib", "libpixelbox_b200.so"))   # PBX_SO: experiment builds only

PBX_OK = 0
ERROR_NAMES = {
    -1: "PBX_E_INVALID", -2: "PBX_E_DIM", -3: "PBX_E_OOM", -4: "PBX_E_CUDA", -5: "PBX_E_NO_DEVICE",
    -6: "PBX_E_CAPACITY", -7: "PBX_E_K", -8: "PBX_E_INTERNAL",
}
PBX_MAX_DIM = 4096
PBX_MAX_K = 2048
DEFAULT_MAX_DIST = 1e3   # DEFAULT_MAX_QUERY_DISTANCE, src/engine.rs:23
DEFAULT_K = 100          # the literal LIMIT of src/engine.rs:381
PBX_FILTER_INCLUDE = 0   # filtered searches: only the listed image ids
PBX_FILTER_EXCLUDE = 1   # ... every row except the listed image ids
PBX_COUNT_FILTER_UNSORTED = 0xFFFFFFFD   # pbx_search_device_filtered: the device filter ids were not sorted

# every symbol include/pixelbox_b200.h declares (tests check the library exports exactly these)
EXPORTS = [
    "pbx_corpus_create", "pbx_corpus_destroy", "pbx_corpus_load", "pbx_corpus_append", "pbx_corpus_flush", "pbx_corpus_append_device",
    "pbx_quantize_device", "pbx_corpus_fill_synthetic", "pbx_corpus_remove", "pbx_sharded_remove",
    "pbx_corpus_replace", "pbx_sharded_replace",
    "pbx_corpus_size", "pbx_corpus_dim", "pbx_corpus_read_rows", "pbx_corpus_synchronize", "pbx_search", "pbx_search_hits", "pbx_search_device",
    "pbx_search_filtered", "pbx_search_device_filtered", "pbx_sharded_search_filtered", "pbx_exchange_search_hits_filtered",
    "pbx_search_page", "pbx_search_device_page", "pbx_sharded_search_page", "pbx_exchange_search_hits_page",
    "pbx_merge_hits", "pbx_merge_hits_device", "pbx_exchange_create", "pbx_exchange_handle", "pbx_exchange_connect",
    "pbx_exchange_allgather_merge", "pbx_exchange_search_hits", "pbx_exchange_destroy",
    "pbx_sharded_create", "pbx_sharded_destroy", "pbx_sharded_load", "pbx_sharded_append", "pbx_sharded_fill_synthetic", "pbx_sharded_size",
    "pbx_sharded_shards", "pbx_sharded_shard", "pbx_sharded_search", "pbx_sharded_search_hits", "pbx_cosine_distance_pairs", "pbx_byte_distance_pairs", "pbx_hamming_distance_pairs", "pbx_quantize", "pbx_get_stats", "pbx_set_candidate_slack",
    "pbx_set_profiling", "pbx_set_batch_min", "pbx_set_scan_ctas_per_sm", "pbx_int8_peak", "pbx_last_error", "pbx_version", "pbx_device_count",
]

HIT_DTYPE = np.dtype([("image_id", "<i8"), ("dist", "<f4"), ("dot", "<i4"), ("norm2", "<i4"), ("flags", "<u4")], align=True)
assert HIT_DTYPE.itemsize == 24


class PbxStats(ctypes.Structure):
    _fields_ = [
        ("rows", ctypes.c_uint64), ("capacity_rows", ctypes.c_uint64), ("dim", ctypes.c_uint32),
        ("row_pitch", ctypes.c_uint32), ("queries", ctypes.c_uint64), ("exact_passes", ctypes.c_uint64),
        ("last_search_ms", ctypes.c_float), ("last_scan_ms", ctypes.c_float), ("last_bytes_scanned", ctypes.c_uint64),
        ("device", ctypes.c_int32), ("sm_count", ctypes.c_int32), ("scan_grid", ctypes.c_int32), ("reserved", ctypes.c_int32),
        ("batched_queries", ctypes.c_uint64),
    ]


class PbxError(RuntimeError):
    def __init__(self, code: int, message: str):
        self.code = code
        self.name = ERROR_NAMES.get(code, f"PBX_E_{code}")
        super().__init__(f"{self.name}: {message}")


_lib = None


def lib() -> ctypes.CDLL:
    """Loads the product library.  Raises if it has not been built (python -m pixelbox_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(f"{SO_PATH} is missing: build it with `python -m pixelbox_b200.build` "
                          "(nvcc, sm_100a). pixelbox_b200 has no CPU or PyTorch fallback.")
    L = ctypes.CDLL(SO_PATH)
    vp, u8p = ctypes.c_void_p, ctypes.c_void_p
    u32, u64, i32, f64 = ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int, ctypes.c_double
    sig = {
        "pbx_corpus_create": (i32, [u32, u64, i32, ctypes.POINTER(vp)]),
        "pbx_corpus_destroy": (None, [vp]),
        "pbx_corpus_load": (i32, [vp, vp, u8p, u64]),
        "pbx_corpus_append": (i32, [vp, vp, u8p, u64]),
        "pbx_corpus_flush": (i32, [vp]),
        "pbx_corpus_append_device": (i32, [vp, vp, vp, u64, vp]),
        "pbx_quantize_device": (i32, [i32, vp, u64, vp, vp]),
        "pbx_corpus_fill_synthetic": (i32, [vp, u64, u64, u64]),
        "pbx_corpus_remove": (i32, [vp, vp, u64, ctypes.POINTER(u64)]),
        "pbx_sharded_remove": (i32, [vp, vp, u64, ctypes.POINTER(u64)]),
        "pbx_corpus_replace": (i32, [vp, vp, u8p, u64, ctypes.POINTER(u64)]),
        "pbx_sharded_replace": (i32, [vp, vp, u8p, u64, ctypes.POINTER(u64)]),
        "pbx_corpus_size": (i32, [vp, ctypes.POINTER(u64)]),
        "pbx_corpus_dim": (i32, [vp, ctypes.POINTER(u32)]),
        "pbx_corpus_read_rows": (i32, [vp, u64, u64, vp, u8p]),
        "pbx_corpus_synchronize": (i32, [vp]),
        "pbx_search": (i32, [vp, u8p, u32, u32, f64, vp, vp, vp, vp, vp]),
        "pbx_search_hits": (i32, [vp, u8p, u32, u32, f64, vp, vp]),
        "pbx_search_device": (i32, [vp, vp, u32, u32, f64, vp, vp, vp]),
        "pbx_search_filtered": (i32, [vp, u8p, u32, u32, f64, vp, vp, vp, vp, vp, vp, u64, u32]),
        "pbx_search_device_filtered": (i32, [vp, vp, u32, u32, f64, vp, vp, vp, vp, u64, u32]),
        "pbx_search_page": (i32, [vp, u8p, u32, u32, f64, vp, vp, u64, u32, vp, vp]),
        "pbx_search_device_page": (i32, [vp, vp, u32, u32, f64, vp, vp, u64, u32, vp, vp, vp]),
        "pbx_merge_hits": (i32, [vp, vp, u32, u32, u32, vp, vp]),
        "pbx_merge_hits_device": (i32, [i32, vp, vp, u32, u32, u32, vp, vp, vp]),
        "pbx_exchange_create": (i32, [i32, u32, u32, u32, u32, ctypes.POINTER(vp)]),
        "pbx_exchange_handle": (i32, [vp, vp]),
        "pbx_exchange_connect": (i32, [vp, vp]),
        "pbx_exchange_allgather_merge": (i32, [vp, vp, u32, u32, vp, vp, vp]),
        "pbx_exchange_search_hits": (i32, [vp, vp, u8p, u32, u32, f64, vp, vp]),
        "pbx_exchange_search_hits_filtered": (i32, [vp, vp, u8p, u32, u32, f64, vp, vp, vp, u64, u32]),
        "pbx_exchange_search_hits_page": (i32, [vp, vp, u8p, u32, u32, f64, vp, vp, u64, u32, vp, vp]),
        "pbx_exchange_destroy": (None, [vp]),
        "pbx_sharded_create": (i32, [u32, u64, vp, i32, ctypes.POINTER(vp)]),
        "pbx_sharded_destroy": (None, [vp]),
        "pbx_sharded_load": (i32, [vp, vp, u8p, u64]),
        "pbx_sharded_append": (i32, [vp, vp, u8p, u64]),
        "pbx_sharded_fill_synthetic": (i32, [vp, u64, u64]),
        "pbx_sharded_size": (i32, [vp, ctypes.POINTER(u64)]),
        "pbx_sharded_shards": (i32, [vp, ctypes.POINTER(u32)]),
        "pbx_sharded_shard": (i32, [vp, u32, ctypes.POINTER(vp)]),
        "pbx_sharded_search": (i32, [vp, u8p, u32, u32, f64, vp, vp, vp, vp, vp]),
        "pbx_sharded_search_hits": (i32, [vp, u8p, u32, u32, f64, vp, vp]),
        "pbx_sharded_search_filtered": (i32, [vp, u8p, u32, u32, f64, vp, vp, vp, vp, vp, vp, u64, u32]),
        "pbx_sharded_search_page": (i32, [vp, u8p, u32, u32, f64, vp, vp, u64, u32, vp, vp]),
        "pbx_cosine_distance_pairs": (i32, [i32, u8p, u8p, u64, u32, vp, vp, vp, vp]),
        "pbx_byte_distance_pairs": (i32, [i32, u8p, u8p, u64, u32, vp, vp]),
        "pbx_hamming_distance_pairs": (i32, [i32, u8p, u8p, u64, u32, vp, vp]),
        "pbx_quantize": (i32, [i32, vp, u64, u8p]),
        "pbx_get_stats": (i32, [vp, ctypes.POINTER(PbxStats)]),
        "pbx_set_candidate_slack": (i32, [vp, u32]),
        "pbx_set_profiling": (i32, [vp, i32]),
        "pbx_set_batch_min": (i32, [vp, u32]),
        "pbx_set_scan_ctas_per_sm": (i32, [vp, u32]),
        "pbx_int8_peak": (i32, [i32, ctypes.POINTER(ctypes.c_double)]),
        "pbx_last_error": (ctypes.c_char_p, []),
        "pbx_version": (ctypes.c_char_p, []),
        "pbx_device_count": (i32, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != PBX_OK:
        raise PbxError(rc, lib().pbx_last_error().decode("utf-8", "replace"))


def filter_args(within, excluding):
    """(ids int64 array, mode) of the `within=` / `excluding=` keywords of the search methods: the image ids a search
    is restricted to, or the ids it must skip.  Passing both is an error."""
    if within is not None and excluding is not None:
        raise ValueError("pass `within` or `excluding`, not both")
    ids = within if within is not None else excluding
    ids = np.ascontiguousarray(np.asarray(ids, dtype=np.int64)).reshape(-1)
    return ids, (PBX_FILTER_INCLUDE if within is not None else PBX_FILTER_EXCLUDE)


def page_filter_args(within, excluding):
    """filter_args for the paged searches, which always take the filter triple: no filter is an empty EXCLUDE set."""
    if within is None and excluding is None:
        return np.zeros(0, np.int64), PBX_FILTER_EXCLUDE
    return filter_args(within, excluding)


def page_cursors(after, nq: int) -> np.ndarray:
    """[nq] pbx_hit cursors of the `after=` keyword of the search methods: one (dist, image_id) per query -- the last
    row of that query's previous page -- or None for its first page ({-inf, INT64_MIN}: no row sorts at or before it).
    A HIT_DTYPE array of nq records (e.g. the last hits of a search_hits call) is taken as is."""
    if isinstance(after, np.ndarray) and after.dtype == HIT_DTYPE:
        cur = np.ascontiguousarray(after.reshape(-1))
        if cur.shape != (nq,):
            raise ValueError(f"after: expected {nq} cursors, got {cur.shape[0]}")
        return cur
    after = list(after)
    if len(after) != nq:
        raise ValueError(f"after: expected one cursor per query ({nq}), got {len(after)}")
    cur = np.zeros(nq, HIT_DTYPE)
    for i, a in enumerate(after):
        if a is None:
            cur[i]["dist"], cur[i]["image_id"] = -np.inf, np.iinfo(np.int64).min
            continue
        if isinstance(a, (str, bytes)) or not hasattr(a, "__len__") or len(a) != 2:
            raise ValueError(f"after[{i}]: expected a (dist, image_id) pair or None, got {a!r}")
        cur[i]["dist"], cur[i]["image_id"] = np.float32(a[0]), int(a[1])
    return cur


def ptr(a) -> ctypes.c_void_p:
    """Raw pointer of a contiguous numpy array (None passes NULL)."""
    if a is None:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(a.ctypes.data)
