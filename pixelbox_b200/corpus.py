"""Corpus: one device-resident shard of the `semantic_hashes` table (src/engine.rs:48) on one B200.

Thin host wrapper over the C ABI (include/pixelbox_b200.h); all compute is in the CUDA library.
"""
from __future__ import annotations

import ctypes
import threading
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from . import _native as nat


class SearchResult(NamedTuple):
    """Rows of one query, ordered by (dist asc, image_id asc) -- what src/engine.rs:384-387 maps."""
    ids: np.ndarray     # int64
    dist: np.ndarray    # float32: the reference's f32 cosine_distance, bit for bit
    dot: np.ndarray     # int32: sum c(q) c(r), c(v) = 2v - 255
    norm2: np.ndarray   # int32: sum c(r)^2


class RangeResult(NamedTuple):
    """The rows of one query within max_dist, ordered by (dist asc, image_id asc), and the exact count of all of them."""
    ids: np.ndarray     # int64
    dist: np.ndarray    # float32, bit for bit
    dot: np.ndarray     # int32
    norm2: np.ndarray   # int32
    total: int          # COUNT(*) of the rows within max_dist (after the cursor, within the filter): >= len(ids)


def _as_u8_2d(a, dim: int, what: str) -> np.ndarray:
    a = np.ascontiguousarray(np.asarray(a, dtype=np.uint8))
    if a.ndim == 1:
        a = a.reshape(1, -1) if a.size else a.reshape(0, dim)
    if a.ndim != 2 or a.shape[1] != dim:
        # the reference would zip-truncate a length mismatch (src/engine.rs:585); the device
        # corpus cannot represent one, so it is an error here (SURVEY.md 8b)
        raise nat.PbxError(-2, f"{what}: expected [n][{dim}] bytes, got shape {tuple(a.shape)}")
    return a


def _hits_results(hits: np.ndarray, cnt: np.ndarray) -> List[SearchResult]:
    """[nq][k] pbx_hit records and [nq] counts -> one SearchResult per query."""
    return [SearchResult(hits[i]["image_id"][:c].copy(), hits[i]["dist"][:c].copy(), hits[i]["dot"][:c].copy(),
                         hits[i]["norm2"][:c].copy()) for i, c in enumerate(cnt.tolist())]


def _remove(fn, handle, image_ids) -> int:
    """fn(handle, ids, n, &rows): a call that takes a list of image ids and returns a row count."""
    ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64)).reshape(-1)
    removed = ctypes.c_uint64(0)
    nat.check(fn(handle, nat.ptr(ids), ids.size, ctypes.byref(removed)))
    return int(removed.value)


def _replace(fn, handle, dim, image_ids, hashes) -> int:
    hashes = _as_u8_2d(hashes, dim, "replace")
    ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64)).reshape(-1)
    if ids.shape != (hashes.shape[0],):
        raise nat.PbxError(-1, "replace: one image_id per hash row required")
    replaced = ctypes.c_uint64(0)
    nat.check(fn(handle, nat.ptr(ids), nat.ptr(hashes), ids.size, ctypes.byref(replaced)))
    return int(replaced.value)


def _search_range(fn, handle, dim: int, size, queries, max_dist, limit, within, excluding, after) -> List[RangeResult]:
    """pbx_search_range / pbx_sharded_search_range (fn), one call per query.  limit = rows wanted per query (None: all of
    them; an answer cut short by rows appended meanwhile is continued from its last row)."""
    fids, mode = nat.page_filter_args(within, excluding)
    q = _as_u8_2d(queries, dim, "search_range")
    nq = q.shape[0]
    cur = None if after is None else nat.page_cursors(after, nq)
    if limit is not None and int(limit) < 0:
        raise ValueError("limit must be >= 0")
    out = []
    offsets = np.zeros(2, np.uint64)
    total = np.zeros(1, np.uint64)
    for i in range(nq):
        cursor = None if cur is None else cur[i:i + 1].copy()
        parts = []
        want = None if limit is None else int(limit)
        first_total = None
        while True:
            cap = size() if want is None else want
            hits = np.empty(cap, nat.HIT_DTYPE)
            nat.check(fn(handle, nat.ptr(q[i:i + 1]), 1, float(max_dist), nat.ptr(cursor), nat.ptr(fids), fids.size, mode,
                         nat.ptr(hits) if cap else None, cap, nat.ptr(offsets), nat.ptr(total)))
            got = hits[:int(offsets[1])]
            parts.append(got)
            if first_total is None:
                first_total = int(total[0])
            if want is not None or len(got) == int(total[0]) or len(got) == 0:
                break
            cursor = got[-1:].copy()                   # rows appended since size() was read: continue after the last row
        rows = np.concatenate(parts) if len(parts) > 1 else parts[0]
        out.append(RangeResult(rows["image_id"].copy(), rows["dist"].copy(), rows["dot"].copy(), rows["norm2"].copy(),
                               max(first_total, len(rows))))
    return out


def _count_within(fn, handle, dim: int, queries, max_dist, within, excluding, after) -> np.ndarray:
    """The exact counts of pbx_search_range with capacity 0, one per query (uint64)."""
    fids, mode = nat.page_filter_args(within, excluding)
    q = _as_u8_2d(queries, dim, "count_within")
    nq = q.shape[0]
    cur = None if after is None else nat.page_cursors(after, nq)
    offsets = np.zeros(nq + 1, np.uint64)
    total = np.zeros(nq, np.uint64)
    nat.check(fn(handle, nat.ptr(q), nq, float(max_dist), nat.ptr(cur), nat.ptr(fids), fids.size, mode, None, 0,
                 nat.ptr(offsets), nat.ptr(total)))
    return total


class Corpus:
    def __init__(self, dim: int, capacity_hint: int = 0, device: int = 0):
        self._h = ctypes.c_void_p(0)
        self.dim = int(dim)
        self.device = int(device)
        nat.check(nat.lib().pbx_corpus_create(self.dim, int(capacity_hint), self.device, ctypes.byref(self._h)))
        self._tls = threading.local()                   # per-thread output buffers of search()
        self._pbx_search = nat.lib().pbx_search

    # -- lifecycle ---------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            nat.lib().pbx_corpus_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __len__(self) -> int:
        n = ctypes.c_uint64(0)
        nat.check(nat.lib().pbx_corpus_size(self._h, ctypes.byref(n)))
        return int(n.value)

    @property
    def handle(self) -> ctypes.c_void_p:
        return self._h

    # -- contents ----------------------------------------------------------------------------
    def load(self, image_ids, hashes) -> None:
        hashes = _as_u8_2d(hashes, self.dim, "load")
        ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64))
        if ids.shape != (hashes.shape[0],):
            raise nat.PbxError(-1, "load: one image_id per hash row required")
        nat.check(nat.lib().pbx_corpus_load(self._h, nat.ptr(ids), nat.ptr(hashes), hashes.shape[0]))

    def append(self, image_ids, hashes) -> None:
        hashes = _as_u8_2d(hashes, self.dim, "append")
        ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64)).reshape(-1)
        if ids.shape != (hashes.shape[0],):
            raise nat.PbxError(-1, "append: one image_id per hash row required")
        nat.check(nat.lib().pbx_corpus_append(self._h, nat.ptr(ids), nat.ptr(hashes), hashes.shape[0]))

    def flush(self) -> None:
        """Uploads the coalesced small appends now (searches do it on their own)."""
        nat.check(nat.lib().pbx_corpus_flush(self._h))

    def append_device(self, d_ids_ptr: int, d_hashes_ptr: int, n: int, stream: Optional[int] = None) -> None:
        """pbx_corpus_append_device: [n] int64 ids and [n][dim] u8 rows already in device memory (raw pointers)."""
        nat.check(nat.lib().pbx_corpus_append_device(self._h, ctypes.c_void_p(d_ids_ptr), ctypes.c_void_p(d_hashes_ptr), int(n),
                                                     ctypes.c_void_p(stream or 0)))

    def remove(self, image_ids) -> int:
        """pbx_corpus_remove: removes every row (pending ones included) whose image_id is listed; returns the number of
        rows removed.  Surviving rows from the tail move into the freed positions (see read_rows)."""
        return _remove(nat.lib().pbx_corpus_remove, self._h, image_ids)

    def replace(self, image_ids, hashes) -> int:
        """pbx_corpus_replace: every row (pending ones included) whose image_id is listed gets the hash listed for it, in
        place (an id listed twice takes its last hash); returns the number of rows written.  Positions do not change."""
        return _replace(nat.lib().pbx_corpus_replace, self._h, self.dim, image_ids, hashes)

    def fill_synthetic(self, n: int, seed: int, first_row: int = 0) -> None:
        nat.check(nat.lib().pbx_corpus_fill_synthetic(self._h, int(n), int(seed), int(first_row)))

    # -- views -------------------------------------------------------------------------------
    def view(self, image_ids) -> "Corpus":
        """pbx_corpus_view_create: a Corpus holding a copy of this corpus' rows whose image_id is listed, kept current by
        this corpus' append / remove / replace / load.  Its searches return what search(..., within=image_ids) returns
        here, at the cost of the view's rows only.  The view is read-only (it follows this corpus); close() it when done.
        It stays searchable if this corpus is closed first."""
        ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64)).reshape(-1)
        v = Corpus.__new__(Corpus)
        v._h = ctypes.c_void_p(0)
        v.dim, v.device = self.dim, self.device
        nat.check(nat.lib().pbx_corpus_view_create(self._h, nat.ptr(ids), ids.size, ctypes.byref(v._h)))
        v._tls = threading.local()
        v._pbx_search = nat.lib().pbx_search
        return v

    def view_add(self, image_ids) -> int:
        """pbx_corpus_view_add (on a view): the parent's rows of the listed ids join it; returns the rows added."""
        return _remove(nat.lib().pbx_corpus_view_add, self._h, image_ids)

    def view_drop(self, image_ids) -> int:
        """pbx_corpus_view_drop (on a view): the rows of the listed ids leave it; returns the rows dropped."""
        return _remove(nat.lib().pbx_corpus_view_drop, self._h, image_ids)

    def read_rows(self, first: int, n: int) -> Tuple[np.ndarray, np.ndarray]:
        ids = np.zeros(n, np.int64)
        rows = np.zeros((n, self.dim), np.uint8)
        nat.check(nat.lib().pbx_corpus_read_rows(self._h, int(first), int(n), nat.ptr(ids), nat.ptr(rows)))
        return ids, rows

    # -- search ------------------------------------------------------------------------------
    def search(self, queries, k: int = nat.DEFAULT_K, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None,
               excluding=None, after=None) -> List[SearchResult]:
        """pbx_search: host buffers in, host buffers out; one SearchResult per query.

        within / excluding (image ids, any order; at most one of them): pbx_search_filtered, the k nearest rows among
        the rows whose id is listed, or among all rows except those -- exactly what a corpus holding only those rows
        would return.

        after (one (dist, image_id) per query, None for a query's first page): pbx_search_page, the k rows that follow
        that position in the (dist, image_id) order -- the next page after a page whose last row was (dist, image_id).
        Combines with within / excluding.

        This is the call the latency of a single interactive query goes through, so the wrapper keeps its own cost
        down: output arrays and their raw pointers are cached per thread and (nq, k), the query pointer is taken from
        the array interface (ndarray.ctypes costs ~1 us per use)."""
        if after is not None:
            return self._search_page(queries, k, max_dist, after, within, excluding)
        if within is not None or excluding is not None:
            return self._search_filtered(queries, k, max_dist, within, excluding)
        if type(queries) is np.ndarray and queries.dtype == np.uint8 and queries.flags.c_contiguous and (
                (queries.ndim == 2 and queries.shape[1] == self.dim) or (queries.ndim == 1 and queries.size == self.dim)):
            q = queries if queries.ndim == 2 else queries.reshape(1, self.dim)
        else:
            q = _as_u8_2d(queries, self.dim, "search")
        nq = q.shape[0]
        k = int(k)
        cache = self._tls.__dict__
        out = cache.get((nq, k))
        if out is None:
            if len(cache) > 64:
                cache.clear()
            ids = np.zeros((nq, k), np.int64)
            dist = np.zeros((nq, k), np.float32)
            dot = np.zeros((nq, k), np.int32)
            n2 = np.zeros((nq, k), np.int32)
            cnt = np.zeros(nq, np.uint32)
            out = cache[(nq, k)] = (ids, dist, dot, n2, cnt, nat.ptr(ids), nat.ptr(dist), nat.ptr(dot), nat.ptr(n2), nat.ptr(cnt))
        ids, dist, dot, n2, cnt, p_ids, p_dist, p_dot, p_n2, p_cnt = out
        rc = self._pbx_search(self._h, q.__array_interface__["data"][0], nq, k, float(max_dist), p_ids, p_dist, p_dot, p_n2, p_cnt)
        if rc:
            nat.check(rc)
        if nq == 1:
            c = int(cnt[0])
            return [SearchResult(ids[0, :c].copy(), dist[0, :c].copy(), dot[0, :c].copy(), n2[0, :c].copy())]
        counts = cnt.tolist()
        return [SearchResult(ids[i, :c].copy(), dist[i, :c].copy(), dot[i, :c].copy(), n2[i, :c].copy()) for i, c in enumerate(counts)]

    def _search_filtered(self, queries, k, max_dist, within, excluding) -> List[SearchResult]:
        fids, mode = nat.filter_args(within, excluding)
        q = _as_u8_2d(queries, self.dim, "search")
        nq, k = q.shape[0], int(k)
        ids, dist, dot, n2 = (np.zeros((nq, k), t) for t in (np.int64, np.float32, np.int32, np.int32))
        cnt = np.zeros(nq, np.uint32)
        nat.check(nat.lib().pbx_search_filtered(self._h, nat.ptr(q), nq, k, float(max_dist), nat.ptr(ids), nat.ptr(dist), nat.ptr(dot),
                                                nat.ptr(n2), nat.ptr(cnt), nat.ptr(fids), fids.size, mode))
        return [SearchResult(ids[i, :c].copy(), dist[i, :c].copy(), dot[i, :c].copy(), n2[i, :c].copy()) for i, c in enumerate(cnt.tolist())]

    def _search_page(self, queries, k, max_dist, after, within, excluding) -> List[SearchResult]:
        fids, mode = nat.page_filter_args(within, excluding)
        q = _as_u8_2d(queries, self.dim, "search")
        nq, k = q.shape[0], int(k)
        cur = nat.page_cursors(after, nq)
        hits = np.zeros((nq, k), nat.HIT_DTYPE)
        cnt = np.zeros(nq, np.uint32)
        nat.check(nat.lib().pbx_search_page(self._h, nat.ptr(q), nq, k, float(max_dist), nat.ptr(cur), nat.ptr(fids), fids.size, mode,
                                            nat.ptr(hits), nat.ptr(cnt)))
        return _hits_results(hits, cnt)

    def search_range(self, queries, max_dist: float = nat.DEFAULT_MAX_DIST, *, limit: Optional[int] = None, within=None,
                     excluding=None, after=None) -> List[RangeResult]:
        """pbx_search_range: every row with dist < max_dist, ordered by (dist, image_id), and the exact count -- the
        similarity query without its LIMIT.  One RangeResult per query.  limit: at most this many rows per query (the
        first ones; total stays exact), None for all.  within / excluding and after as in search()."""
        return _search_range(nat.lib().pbx_search_range, self._h, self.dim, self.__len__, queries, max_dist, limit, within,
                             excluding, after)

    def count_within(self, queries, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None, excluding=None, after=None) -> np.ndarray:
        """pbx_search_range with capacity 0: COUNT(*) of the rows with dist < max_dist, per query (uint64 array)."""
        return _count_within(nat.lib().pbx_search_range, self._h, self.dim, queries, max_dist, within, excluding, after)

    def search_hits(self, queries, k: int = nat.DEFAULT_K, max_dist: float = nat.DEFAULT_MAX_DIST) -> Tuple[np.ndarray, np.ndarray]:
        """pbx_search_hits: ([nq][k] pbx_hit records, [nq] counts) -- the per-shard half of a sharded search."""
        q = _as_u8_2d(queries, self.dim, "search_hits")
        nq = q.shape[0]
        hits = np.zeros((nq, k), nat.HIT_DTYPE)
        cnt = np.zeros(nq, np.uint32)
        nat.check(nat.lib().pbx_search_hits(self._h, nat.ptr(q), nq, int(k), float(max_dist), nat.ptr(hits), nat.ptr(cnt)))
        return hits, cnt

    def search_device(self, d_queries_ptr: int, nq: int, k: int, max_dist: float, d_hits_ptr: int, d_count_ptr: int,
                      stream: Optional[int] = None) -> None:
        """pbx_search_device: raw device pointers, enqueued on `stream`, no host sync.

        `stream` is a cudaStream_t value (e.g. torch.cuda.current_stream().cuda_stream); 0 means the
        legacy default stream, as it does in torch; None means the corpus' own stream (wait for it
        with synchronize())."""
        if stream is None:
            stream = 0                      # NULL -> the corpus' own stream
        elif stream == 0:
            stream = 1                      # cudaStreamLegacy
        nat.check(nat.lib().pbx_search_device(self._h, ctypes.c_void_p(d_queries_ptr), int(nq), int(k), float(max_dist),
                                              ctypes.c_void_p(d_hits_ptr), ctypes.c_void_p(d_count_ptr),
                                              ctypes.c_void_p(stream)))

    def search_device_filtered(self, d_queries_ptr: int, nq: int, k: int, max_dist: float, d_hits_ptr: int, d_count_ptr: int,
                               d_filter_ids_ptr: int, n_filter: int, mode: int = nat.PBX_FILTER_INCLUDE,
                               stream: Optional[int] = None) -> None:
        """pbx_search_device_filtered: search_device restricted by [n_filter] int64 image ids at d_filter_ids_ptr (device
        memory, sorted ascending; mode PBX_FILTER_INCLUDE or PBX_FILTER_EXCLUDE).  Unsorted ids are reported on the
        device: every count of the call becomes PBX_COUNT_FILTER_UNSORTED."""
        if stream is None:
            stream = 0
        elif stream == 0:
            stream = 1
        nat.check(nat.lib().pbx_search_device_filtered(self._h, ctypes.c_void_p(d_queries_ptr), int(nq), int(k), float(max_dist),
                                                       ctypes.c_void_p(d_hits_ptr), ctypes.c_void_p(d_count_ptr), ctypes.c_void_p(stream),
                                                       ctypes.c_void_p(d_filter_ids_ptr), int(n_filter), int(mode)))

    def search_device_page(self, d_queries_ptr: int, nq: int, k: int, max_dist: float, d_hits_ptr: int, d_count_ptr: int,
                           d_after_ptr: int = 0, d_filter_ids_ptr: int = 0, n_filter: int = 0, mode: int = nat.PBX_FILTER_EXCLUDE,
                           stream: Optional[int] = None) -> None:
        """pbx_search_device_page: search_device for the rows after [nq] pbx_hit cursors at d_after_ptr (device memory, read
        in stream order; 0 = first pages), optionally filtered as in search_device_filtered (n_filter = 0 with
        PBX_FILTER_EXCLUDE: no filter).  The cursors may be the previous call's records (slot count - 1 of each query):
        pages chain without a host read.  A NaN cursor dist gives that query count 0."""
        if stream is None:
            stream = 0
        elif stream == 0:
            stream = 1
        nat.check(nat.lib().pbx_search_device_page(self._h, ctypes.c_void_p(d_queries_ptr), int(nq), int(k), float(max_dist),
                                                   ctypes.c_void_p(d_after_ptr), ctypes.c_void_p(d_filter_ids_ptr), int(n_filter),
                                                   int(mode), ctypes.c_void_p(d_hits_ptr), ctypes.c_void_p(d_count_ptr),
                                                   ctypes.c_void_p(stream)))

    def synchronize(self) -> None:
        """Waits for everything enqueued on the corpus' own stream."""
        nat.check(nat.lib().pbx_corpus_synchronize(self._h))

    # -- diagnostics -------------------------------------------------------------------------
    def stats(self) -> nat.PbxStats:
        s = nat.PbxStats()
        nat.check(nat.lib().pbx_get_stats(self._h, ctypes.byref(s)))
        return s

    def set_candidate_slack(self, slack: int) -> None:
        nat.check(nat.lib().pbx_set_candidate_slack(self._h, int(slack)))

    def set_profiling(self, enabled: bool) -> None:
        """Record CUDA events around searches (stats().last_search_ms / last_scan_ms); off by default."""
        nat.check(nat.lib().pbx_set_profiling(self._h, 1 if enabled else 0))

    def set_batch_min(self, n: int) -> None:
        """Calls with at least n queries use the tensor-core path (0 = default 2, 0xFFFFFFFF = never)."""
        nat.check(nat.lib().pbx_set_batch_min(self._h, int(n)))

    def set_scan_ctas_per_sm(self, n: int) -> None:
        nat.check(nat.lib().pbx_set_scan_ctas_per_sm(self._h, int(n)))


class MultiDeviceCorpus:
    """pbx_sharded_*: the table row-sharded over several GPUs of this box by ONE process (one worker thread and
    stream per shard inside the library, merge on the first device).  Same results as one Corpus holding all rows."""

    def __init__(self, dim: int, devices: Sequence[int], capacity_hint: int = 0):
        self._h = ctypes.c_void_p(0)
        self.dim = int(dim)
        self.devices = [int(d) for d in devices]
        arr = (ctypes.c_int * len(self.devices))(*self.devices)
        nat.check(nat.lib().pbx_sharded_create(self.dim, int(capacity_hint), ctypes.cast(arr, ctypes.c_void_p), len(self.devices), ctypes.byref(self._h)))

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            nat.lib().pbx_sharded_destroy(self._h)
            self._h = ctypes.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __len__(self) -> int:
        n = ctypes.c_uint64(0)
        nat.check(nat.lib().pbx_sharded_size(self._h, ctypes.byref(n)))
        return int(n.value)

    def load(self, image_ids, hashes) -> None:
        hashes = _as_u8_2d(hashes, self.dim, "load")
        ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64))
        if ids.shape != (hashes.shape[0],):
            raise nat.PbxError(-1, "load: one image_id per hash row required")
        nat.check(nat.lib().pbx_sharded_load(self._h, nat.ptr(ids), nat.ptr(hashes), hashes.shape[0]))

    def append(self, image_ids, hashes) -> None:
        hashes = _as_u8_2d(hashes, self.dim, "append")
        ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64)).reshape(-1)
        if ids.shape != (hashes.shape[0],):
            raise nat.PbxError(-1, "append: one image_id per hash row required")
        nat.check(nat.lib().pbx_sharded_append(self._h, nat.ptr(ids), nat.ptr(hashes), hashes.shape[0]))

    def remove(self, image_ids) -> int:
        """pbx_sharded_remove: every shard removes the listed ids; returns the total number of rows removed."""
        return _remove(nat.lib().pbx_sharded_remove, self._h, image_ids)

    def replace(self, image_ids, hashes) -> int:
        """pbx_sharded_replace: every shard replaces the hashes of the listed ids; returns the total number of rows written."""
        return _replace(nat.lib().pbx_sharded_replace, self._h, self.dim, image_ids, hashes)

    def fill_synthetic(self, rows_per_shard: int, seed: int) -> None:
        nat.check(nat.lib().pbx_sharded_fill_synthetic(self._h, int(rows_per_shard), int(seed)))

    def view(self, image_ids) -> "MultiDeviceCorpus":
        """pbx_sharded_view_create: one view per shard (see Corpus.view); searched like this corpus."""
        ids = np.ascontiguousarray(np.asarray(image_ids, dtype=np.int64)).reshape(-1)
        v = MultiDeviceCorpus.__new__(MultiDeviceCorpus)
        v._h = ctypes.c_void_p(0)
        v.dim, v.devices = self.dim, list(self.devices)
        nat.check(nat.lib().pbx_sharded_view_create(self._h, nat.ptr(ids), ids.size, ctypes.byref(v._h)))
        return v

    def view_add(self, image_ids) -> int:
        """pbx_sharded_view_add (on a view): returns the rows added over all shards."""
        return _remove(nat.lib().pbx_sharded_view_add, self._h, image_ids)

    def view_drop(self, image_ids) -> int:
        """pbx_sharded_view_drop (on a view): returns the rows dropped over all shards."""
        return _remove(nat.lib().pbx_sharded_view_drop, self._h, image_ids)

    def shard_stats(self, index: int) -> nat.PbxStats:
        h = ctypes.c_void_p(0)
        nat.check(nat.lib().pbx_sharded_shard(self._h, int(index), ctypes.byref(h)))
        s = nat.PbxStats()
        nat.check(nat.lib().pbx_get_stats(h, ctypes.byref(s)))
        return s

    def set_candidate_slack(self, slack: int) -> None:
        for i in range(len(self.devices)):
            h = ctypes.c_void_p(0)
            nat.check(nat.lib().pbx_sharded_shard(self._h, i, ctypes.byref(h)))
            nat.check(nat.lib().pbx_set_candidate_slack(h, int(slack)))

    def search(self, queries, k: int = nat.DEFAULT_K, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None,
               excluding=None, after=None) -> List[SearchResult]:
        """pbx_sharded_search; within / excluding and after as in Corpus.search (pbx_sharded_search_filtered,
        pbx_sharded_search_page)."""
        if after is not None:
            fids, mode = nat.page_filter_args(within, excluding)
            q = _as_u8_2d(queries, self.dim, "search")
            nq, k = q.shape[0], int(k)
            cur = nat.page_cursors(after, nq)
            hits = np.zeros((nq, k), nat.HIT_DTYPE)
            cnt = np.zeros(nq, np.uint32)
            nat.check(nat.lib().pbx_sharded_search_page(self._h, nat.ptr(q), nq, k, float(max_dist), nat.ptr(cur), nat.ptr(fids), fids.size,
                                                        mode, nat.ptr(hits), nat.ptr(cnt)))
            return _hits_results(hits, cnt)
        filtered = within is not None or excluding is not None
        if filtered:
            fids, mode = nat.filter_args(within, excluding)
        q = _as_u8_2d(queries, self.dim, "search")
        nq, k = q.shape[0], int(k)
        ids = np.zeros((nq, k), np.int64)
        dist = np.zeros((nq, k), np.float32)
        dot = np.zeros((nq, k), np.int32)
        n2 = np.zeros((nq, k), np.int32)
        cnt = np.zeros(nq, np.uint32)
        if filtered:
            nat.check(nat.lib().pbx_sharded_search_filtered(self._h, nat.ptr(q), nq, k, float(max_dist), nat.ptr(ids), nat.ptr(dist),
                                                            nat.ptr(dot), nat.ptr(n2), nat.ptr(cnt), nat.ptr(fids), fids.size, mode))
        else:
            nat.check(nat.lib().pbx_sharded_search(self._h, nat.ptr(q), nq, k, float(max_dist), nat.ptr(ids), nat.ptr(dist), nat.ptr(dot),
                                                   nat.ptr(n2), nat.ptr(cnt)))
        return [SearchResult(ids[i, :c].copy(), dist[i, :c].copy(), dot[i, :c].copy(), n2[i, :c].copy()) for i, c in enumerate(cnt.tolist())]

    def search_range(self, queries, max_dist: float = nat.DEFAULT_MAX_DIST, *, limit: Optional[int] = None, within=None,
                     excluding=None, after=None) -> List[RangeResult]:
        """pbx_sharded_search_range, as Corpus.search_range."""
        return _search_range(nat.lib().pbx_sharded_search_range, self._h, self.dim, self.__len__, queries, max_dist, limit,
                             within, excluding, after)

    def count_within(self, queries, max_dist: float = nat.DEFAULT_MAX_DIST, *, within=None, excluding=None, after=None) -> np.ndarray:
        """pbx_sharded_search_range with capacity 0, as Corpus.count_within."""
        return _count_within(nat.lib().pbx_sharded_search_range, self._h, self.dim, queries, max_dist, within, excluding, after)


def merge_hits(gathered: np.ndarray, counts: np.ndarray, k: int) -> Tuple[np.ndarray, np.ndarray]:
    """pbx_merge_hits: gathered [n_shards][nq][k] records + counts [n_shards][nq] -> global ([nq][k], [nq])."""
    gathered = np.ascontiguousarray(gathered, dtype=nat.HIT_DTYPE)
    counts = np.ascontiguousarray(counts, dtype=np.uint32)
    n_shards, nq = counts.shape
    assert gathered.shape == (n_shards, nq, k), (gathered.shape, (n_shards, nq, k))
    out = np.zeros((nq, k), nat.HIT_DTYPE)
    cnt = np.zeros(nq, np.uint32)
    nat.check(nat.lib().pbx_merge_hits(nat.ptr(gathered), nat.ptr(counts), n_shards, nq, int(k), nat.ptr(out), nat.ptr(cnt)))
    return out, cnt


def cosine_distance_pairs(a, b, device: int = 0):
    """pbx_cosine_distance_pairs: the reference's cosine_distance (src/engine.rs:572-588) on the GPU for
    explicit pairs; returns (dist f32, dot i32, norm2_a i32, norm2_b i32)."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.uint8))
    b = np.ascontiguousarray(np.asarray(b, dtype=np.uint8))
    if a.ndim == 1:
        a, b = a.reshape(1, -1), b.reshape(1, -1)
    if a.shape != b.shape:
        raise nat.PbxError(-2, f"pair shapes differ: {a.shape} vs {b.shape}")
    n, d = a.shape
    dist = np.zeros(n, np.float32)
    dot = np.zeros(n, np.int32)
    na = np.zeros(n, np.int32)
    nb = np.zeros(n, np.int32)
    nat.check(nat.lib().pbx_cosine_distance_pairs(int(device), nat.ptr(a), nat.ptr(b), n, d, nat.ptr(dist), nat.ptr(dot),
                                                  nat.ptr(na), nat.ptr(nb)))
    return dist, dot, na, nb


def _pairs(a, b):
    a = np.ascontiguousarray(np.asarray(a, dtype=np.uint8))
    b = np.ascontiguousarray(np.asarray(b, dtype=np.uint8))
    if a.ndim == 1:
        a, b = a.reshape(1, -1), b.reshape(1, -1)
    if a.shape != b.shape:
        raise nat.PbxError(-2, f"pair shapes differ: {a.shape} vs {b.shape}")
    return a, b


def byte_distance_pairs(a, b, device: int = 0):
    """pbx_byte_distance_pairs: the reference's byte_distance (src/engine.rs:590-592); returns (dist f32, L1 sum u32)."""
    a, b = _pairs(a, b)
    n, d = a.shape
    dist, l1 = np.zeros(n, np.float32), np.zeros(n, np.uint32)
    nat.check(nat.lib().pbx_byte_distance_pairs(int(device), nat.ptr(a), nat.ptr(b), n, d, nat.ptr(dist), nat.ptr(l1)))
    return dist, l1


def hamming_distance_pairs(a, b, device: int = 0):
    """pbx_hamming_distance_pairs: the reference's hamming_distance (src/engine.rs:594-604, u8 sum wrapping as in a
    release build); returns (dist f32, true differing bits u32)."""
    a, b = _pairs(a, b)
    n, d = a.shape
    dist, bits = np.zeros(n, np.float32), np.zeros(n, np.uint32)
    nat.check(nat.lib().pbx_hamming_distance_pairs(int(device), nat.ptr(a), nat.ptr(b), n, d, nat.ptr(dist), nat.ptr(bits)))
    return dist, bits


def quantize_device(d_in_ptr: int, n: int, d_out_ptr: int, device: int = 0, stream: Optional[int] = None) -> None:
    """pbx_quantize_device: n floats at d_in_ptr -> n bytes at d_out_ptr, both device memory; asynchronous on `stream`."""
    nat.check(nat.lib().pbx_quantize_device(int(device), ctypes.c_void_p(d_in_ptr), int(n), ctypes.c_void_p(d_out_ptr), ctypes.c_void_p(stream or 0)))


def quantize(embeddings, device: int = 0) -> np.ndarray:
    """pbx_quantize: the reference's f32 -> u8 encoder (src/image_hashes/efficientnet.rs:39) on the GPU."""
    f = np.ascontiguousarray(np.asarray(embeddings, dtype=np.float32))
    out = np.zeros(f.shape, np.uint8)
    nat.check(nat.lib().pbx_quantize(int(device), nat.ptr(f), f.size, nat.ptr(out)))
    return out
