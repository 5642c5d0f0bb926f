"""Paged searches without a GPU: the C ABI's argument checks (NULL outputs, NaN cursors, k, the filter rules), the
`after=` checks of the Python wrappers, and the numpy page oracle (tests/page_oracle.py) against the keyset SQL in
SQLite, ties and the 999999 plateau included."""
import ctypes
import sqlite3

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus
from tests import page_oracle, sqlite_oracle

INT64_MIN, INT64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


def _err():
    return nat.lib().pbx_last_error().decode()


def _host_calls(after, k=10, fids=None, n_filter=0, mode=nat.PBX_FILTER_EXCLUDE, out=True, handle=None):
    """The three host-form page entry points (NULL handles unless given) with valid buffers otherwise."""
    L = nat.lib()
    q = np.zeros((1, 8), np.uint8)
    hits, cnt = np.zeros(max(k, 1), nat.HIT_DTYPE), np.zeros(1, np.uint32)
    hp, cp = (nat.ptr(hits), nat.ptr(cnt)) if out else (None, None)
    ap = nat.ptr(after) if after is not None else None
    fp = nat.ptr(fids) if fids is not None else None
    yield L.pbx_search_page(handle, nat.ptr(q), 1, k, 1e3, ap, fp, n_filter, mode, hp, cp)
    yield L.pbx_sharded_search_page(handle, nat.ptr(q), 1, k, 1e3, ap, fp, n_filter, mode, hp, cp)
    yield L.pbx_exchange_search_hits_page(handle, None, nat.ptr(q), 1, k, 1e3, ap, fp, n_filter, mode, hp, cp)


def cursor(d, i):
    c = np.zeros(1, nat.HIT_DTYPE)
    c[0]["dist"], c[0]["image_id"] = d, i
    return c


def test_null_handles_are_invalid():
    for rc in _host_calls(cursor(0.5, 3)):
        assert rc == -1 and "NULL" in _err()
    assert nat.lib().pbx_search_device_page(None, None, 1, 10, 1e3, None, None, 0, nat.PBX_FILTER_EXCLUDE, None, None, None) == -1


def test_nan_cursor_is_invalid():
    for rc in _host_calls(cursor(np.nan, 3)):
        assert rc == -1 and "NaN" in _err()


def test_filter_rules_are_those_of_the_filtered_searches():
    fids = np.array([1], np.int64)
    for rc in _host_calls(cursor(0.5, 3), fids=None, n_filter=5, mode=nat.PBX_FILTER_INCLUDE):
        assert rc == -1 and "filter_ids is NULL" in _err()
    for mode in (2, 0xFFFFFFFF):
        for rc in _host_calls(cursor(0.5, 3), fids=fids, n_filter=1, mode=mode):
            assert rc == -1 and "unknown filter mode" in _err()
    for rc in _host_calls(cursor(0.5, 3), fids=fids, n_filter=0xFFFFF001, mode=nat.PBX_FILTER_INCLUDE):
        assert rc == -1 and "PBX_MAX_ROWS" in _err()
    rc = nat.lib().pbx_search_device_page(None, None, 1, 10, 1e3, None, None, 3, nat.PBX_FILTER_INCLUDE, None, None, None)
    assert rc == -1 and "filter_ids is NULL" in _err()


def test_k_and_outputs_need_no_device():
    # a NULL corpus fails before k or the outputs are looked at; what the calls do with a corpus is checked on the GPU
    for rc in _host_calls(None, k=0):
        assert rc == -1
    for rc in _host_calls(None, out=False):
        assert rc == -1


def test_after_shape_checks():
    assert nat.page_cursors([None, (0.25, 7)], 2)["image_id"].tolist() == [INT64_MIN, 7]
    cur = nat.page_cursors([None], 1)
    assert np.isneginf(cur[0]["dist"]) and cur[0]["image_id"] == INT64_MIN
    assert nat.page_cursors(np.zeros(3, nat.HIT_DTYPE), 3).shape == (3,)
    for bad, nq in (([None], 2), ([(0.5, 1)] * 3, 2), ((0.5, 3), 1), ([(0.5,)], 1), ([(0.5, 1, 2)], 1), (["ab"], 1),
                    (np.zeros(2, nat.HIT_DTYPE), 3)):
        with pytest.raises(ValueError):
            nat.page_cursors(bad, nq)
    ids, mode = nat.page_filter_args(None, None)
    assert ids.size == 0 and mode == nat.PBX_FILTER_EXCLUDE
    with pytest.raises(ValueError):
        nat.page_filter_args([1], [2])
    # the wrappers check before any native call: instances without a device handle are enough
    for cls in (Corpus, MultiDeviceCorpus):
        obj = cls.__new__(cls)
        obj._h, obj.dim = ctypes.c_void_p(0), 8
        with pytest.raises(ValueError):
            obj.search(np.zeros((2, 8), np.uint8), 10, after=[None])
        with pytest.raises(ValueError):
            obj.search(np.zeros(8, np.uint8), 10, after=[None], within=[1], excluding=[2])


# ---- the numpy page oracle against the keyset SQL --------------------------------------------------------------------
KEYSET_SQL = """SELECT image_id, cosine_distance(?, hash) AS dist FROM semantic_hashes
                WHERE dist < ? AND (dist > ? OR (dist = ? AND image_id > ?)) {filt}
                ORDER BY dist ASC, image_id ASC LIMIT ?"""


def keyset(conn, q, k, max_dist, cur, within=None):
    filt = "" if within is None else f"AND image_id IN ({','.join(str(int(i)) for i in within)})"
    d0, id0 = (float("-inf"), int(INT64_MIN)) if cur is None else (float(np.float32(cur[0])), int(cur[1]))
    rows = conn.execute(KEYSET_SQL.format(filt=filt), (bytes(q), float(max_dist), d0, d0, id0, int(k))).fetchall()
    return [r[0] for r in rows], np.array([r[1] for r in rows], np.float64).astype(np.float32)


def table(d, seed):
    rng = np.random.default_rng(seed)
    n = 400
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    rows[10:40] = rows[10]                                  # a tie of identical rows
    rows[300:330] = 255 - rows[300]                         # antipodes of one row: a tie on the plateau for that query
    ids = rng.permutation(np.arange(-n // 2, n - n // 2)).astype(np.int64) * 7
    ids[0], ids[1] = INT64_MIN, INT64_MAX
    return rows, ids


@pytest.mark.parametrize("d", [8, 64])
def test_page_oracle_is_the_keyset_sql(d):
    rows, ids = table(d, 40 + d)
    conn = sqlite3.connect(":memory:")
    conn.execute(sqlite_oracle.HASH_TABLE_SCHEMA_V1)
    conn.executemany("INSERT INTO semantic_hashes (image_id, hash) VALUES (?, ?)", [(int(i), bytes(h)) for i, h in zip(ids, rows)])
    sqlite_oracle.register(conn)
    within = ids[::3]
    allowed = np.isin(ids, within)
    for q in (rows[10], rows[300], rows[77]):
        dist = oracle.all_distances(rows, q)
        for max_dist, k in ((1e3, 7), (1e7, 50), (0.9, 13)):
            for filtered in (False, True):
                cur, depth = None, 0
                full, _ = page_oracle.order(rows, ids, q, max_dist, allowed if filtered else None, dist)
                while True:
                    want_ids, want_dist = keyset(conn, q, k, max_dist, cur, within if filtered else None)
                    got = page_oracle.page(rows, ids, q, k, max_dist, cur, allowed if filtered else None, dist)
                    assert list(got[0]) == want_ids and np.array_equal(got[1].view(np.uint32), want_dist.view(np.uint32))
                    assert list(got[0]) == list(ids[full[depth:depth + k]])           # pages concatenate to one deep order
                    for i, row_id in enumerate(got[0]):
                        r = rows[np.nonzero(ids == row_id)[0][0]]
                        assert (got[2][i], got[3][i]) == oracle.int_terms(q, r)[::2]
                    if len(want_ids) < k:
                        break
                    cur, depth = (got[1][-1], got[0][-1]), depth + k
        # cursors that are no row: between two dists, past every row, before every row
        for cur in ((dist[5], -3), (np.float32(np.inf), INT64_MIN), (np.float32(-np.inf), INT64_MIN), (np.float32(-1.0), 0),
                    (np.float32(999999.0), ids[300]), (np.float32(999999.0), INT64_MIN)):
            want_ids, _ = keyset(conn, q, 1000, 1e7, cur)
            assert list(page_oracle.page(rows, ids, q, 1000, 1e7, cur, dists=dist)[0]) == want_ids
