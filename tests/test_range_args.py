"""Range searches without a GPU: the C ABI's argument checks, the checks of the Python wrappers, the numpy range oracle
(tests/range_oracle.py) against the similarity SQL without its LIMIT and its COUNT(*) in SQLite, and the two kappa cuts
of range_cut (page.cuh) restated in numpy: a row classified certainly inside has dist < max_dist, one classified
certainly outside does not."""
import ctypes
import sqlite3

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus
from tests import range_oracle, sqlite_oracle

INT64_MIN, INT64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


def _err():
    return nat.lib().pbx_last_error().decode()


def cursor(d, i):
    c = np.zeros(1, nat.HIT_DTYPE)
    c[0]["dist"], c[0]["image_id"] = d, i
    return c


def _calls(after=None, fids=None, n_filter=0, mode=nat.PBX_FILTER_EXCLUDE, capacity=10, hits=True, offsets=True, total=True):
    """Both range entry points with NULL handles and otherwise valid buffers."""
    L = nat.lib()
    q = np.zeros((1, 8), np.uint8)
    h = np.zeros(max(capacity, 1), nat.HIT_DTYPE)
    off, tot = np.zeros(2, np.uint64), np.zeros(1, np.uint64)
    args = (nat.ptr(q), 1, 1e3, nat.ptr(after) if after is not None else None, nat.ptr(fids) if fids is not None else None,
            n_filter, mode, nat.ptr(h) if hits else None, capacity, nat.ptr(off) if offsets else None, nat.ptr(tot) if total else None)
    yield L.pbx_search_range(None, *args)
    yield L.pbx_sharded_search_range(None, *args)


def test_null_handles_and_outputs_are_invalid():
    for kw in ({}, {"hits": False}, {"offsets": False}, {"total": False}, {"capacity": 0, "hits": False}):
        for rc in _calls(cursor(0.5, 3), **kw):
            assert rc == -1 and "NULL" in _err()


def test_nan_cursor_is_invalid():
    for rc in _calls(cursor(np.nan, 3)):
        assert rc == -1 and "NaN" in _err()


def test_filter_rules_are_those_of_the_filtered_searches():
    fids = np.array([1], np.int64)
    for rc in _calls(fids=None, n_filter=5, mode=nat.PBX_FILTER_INCLUDE):
        assert rc == -1 and "filter_ids is NULL" in _err()
    for mode in (2, 0xFFFFFFFF):
        for rc in _calls(fids=fids, n_filter=1, mode=mode):
            assert rc == -1 and "unknown filter mode" in _err()
    for rc in _calls(fids=fids, n_filter=0xFFFFF001, mode=nat.PBX_FILTER_INCLUDE):
        assert rc == -1 and "PBX_MAX_ROWS" in _err()


def test_wrapper_checks_need_no_device():
    for cls in (Corpus, MultiDeviceCorpus):
        obj = cls.__new__(cls)
        obj._h, obj.dim = ctypes.c_void_p(0), 8
        q = np.zeros((2, 8), np.uint8)
        with pytest.raises(ValueError):
            obj.search_range(q, 0.5, after=[None])
        with pytest.raises(ValueError):
            obj.count_within(q, 0.5, after=[None, None, None])
        with pytest.raises(ValueError):
            obj.search_range(q, 0.5, within=[1], excluding=[2])
        with pytest.raises(ValueError):
            obj.search_range(q, 0.5, limit=-1)
        with pytest.raises(nat.PbxError):
            obj.count_within(np.zeros((1, 9), np.uint8), 0.5)


# ---- the numpy range oracle against the SQL without LIMIT ------------------------------------------------------------
RANGE_SQL = """SELECT image_id, cosine_distance(?, hash) AS dist FROM semantic_hashes
               WHERE dist < ? {cur} {filt}
               ORDER BY dist ASC"""
COUNT_SQL = """SELECT COUNT(*) FROM (SELECT image_id, cosine_distance(?, hash) AS dist FROM semantic_hashes
               WHERE dist < ? {cur} {filt})"""


def sql_range(conn, q, max_dist, cur=None, within=None):
    filt = "" if within is None else f"AND image_id IN ({','.join(str(int(i)) for i in within)})"
    args = [bytes(q), float(max_dist)]
    c = ""
    if cur is not None:
        c = "AND (dist > ? OR (dist = ? AND image_id > ?))"
        d0 = float(np.float32(cur[0]))
        args += [d0, d0, int(cur[1])]
    rows = conn.execute(RANGE_SQL.format(cur=c, filt=filt), args).fetchall()
    count = conn.execute(COUNT_SQL.format(cur=c, filt=filt), args).fetchone()[0]
    return [r[0] for r in rows], np.array([r[1] for r in rows], np.float64).astype(np.float32), count


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
def test_range_oracle_is_the_sql_without_limit(d):
    rows, ids = table(d, 70 + d)
    conn = sqlite3.connect(":memory:")
    conn.execute(sqlite_oracle.HASH_TABLE_SCHEMA_V1)
    conn.executemany("INSERT INTO semantic_hashes (image_id, hash) VALUES (?, ?)", [(int(i), bytes(h)) for i, h in zip(ids, rows)])
    sqlite_oracle.register(conn)
    within = ids[::3]
    allowed = np.isin(ids, within)
    for q in (rows[10], rows[300], rows[77]):
        dist = oracle.all_distances(rows, q)
        some = float(np.sort(dist)[len(dist) // 3])
        radii = [0.0, -0.5, -1.0, 999999.0, float(np.nextafter(np.float32(999999.0), np.float32(np.inf))), 999999.5, 1e3,
                 np.inf, np.nan, some, float(np.nextafter(np.float32(some), np.float32(np.inf))), 0.9]
        for max_dist in radii:
            for filtered in (False, True):
                for cur in (None, (some, 0), (np.float32(999999.0), ids[305]), (np.float32(-np.inf), INT64_MIN)):
                    want_ids, want_dist, count = sql_range(conn, q, max_dist, cur, within if filtered else None)
                    got = range_oracle.answer(rows, ids, q, max_dist, cur, allowed if filtered else None, dist)
                    assert list(got[0]) == want_ids and len(want_ids) == count
                    assert np.array_equal(got[1].view(np.uint32), want_dist.view(np.uint32))
        # identical rows are inside at max_dist = 0 (dist -1.19e-7); a NaN radius admits nothing; above 999999 everything
        if q is rows[10]:
            assert len(range_oracle.answer(rows, ids, q, 0.0, dists=dist)[0]) == 30
        assert len(range_oracle.answer(rows, ids, q, np.nan, dists=dist)[0]) == 0
        assert len(range_oracle.answer(rows, ids, q, 1e6, dists=dist)[0]) == len(rows)


# ---- the cuts --------------------------------------------------------------------------------------------------------
def cut_case(rng, d, kind, n=2000):
    if kind == "uniform":
        rows = rng.integers(0, 256, size=(n, d))
    elif kind == "wild":        # almost no norm, maximal norm and dark rows side by side
        rows = rng.integers(0, 256, size=(n, d))
        rows[: n // 4] = rng.integers(127, 129, size=(n // 4, d))
        rows[n // 4: n // 2] = rng.integers(0, 2, size=(n // 4, d)) * 255
        rows[n // 2: 3 * n // 4] = rng.integers(0, 40, size=(n // 4, d))
    else:                       # "near": a near-duplicate cluster around the query
        rows = np.clip(rng.integers(0, 256, size=(1, d)) + rng.integers(-2, 3, size=(n, d)), 0, 255)
    q = rows[rng.integers(0, n)].copy()
    if rng.random() < 0.5:
        q = np.clip(q + rng.integers(-10, 11, size=d), 0, 255)
    if rng.random() < 0.3:
        q = 255 - q
    return rows.astype(np.uint8), q.astype(np.uint8)


@pytest.mark.parametrize("d", [8, 64, 100, 256, 1024])
@pytest.mark.parametrize("kind", ["uniform", "wild", "near"])
def test_cuts_classify_rows_correctly(d, kind):
    rng = np.random.default_rng([d, ["uniform", "wild", "near"].index(kind)])
    margin = range_oracle.certificate_margin(d)
    inside = outside = 0
    for _ in range(3):
        rows, q = cut_case(rng, d, kind)
        dist = oracle.all_distances(rows, q)
        kap = range_oracle.kappas(rows, q)
        # radii at the exact f32 dist of rows and their neighbours, the plateau edge, and the degenerate ones
        picks = dist[rng.integers(0, len(dist), 40)]
        radii = set()
        for x in picks:
            for y in (x, np.nextafter(x, np.float32(np.inf)), np.nextafter(x, np.float32(-np.inf))):
                radii.add(float(y))
        radii |= {0.0, -1.0, -0.999, -2.0, 999999.0, 999999.5, 1e7, np.inf, -np.inf, float("nan"), 1e-7, -1.2e-7}
        for max_dist in radii:
            m = range_oracle.dist_bound(max_dist)
            lo, hi = range_oracle.range_cut(m, margin)
            truth = dist.astype(np.float64) < max_dist
            assert np.array_equal(truth, dist < m) or np.isnan(max_dist)      # the f32 bound is the f64 comparison
            assert truth[kap > hi].all(), (max_dist, d, kind)
            assert not truth[kap < lo].any(), (max_dist, d, kind)
            inside += int((kap > hi).sum())
            outside += int((kap < lo).sum())
    assert inside > 0 and outside > 0
