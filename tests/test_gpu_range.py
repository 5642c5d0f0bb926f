"""Range searches (pbx_search_range, Corpus.search_range / count_within and their twins): every row with dist < max_dist
in (dist, image_id) order and the exact count -- ids, order, dist bit for bit, dot, norm2 and total, compared with the
numpy range oracle over the whole corpus (tests/range_oracle.py, checked against the SQL without LIMIT on the CPU)."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200 import synth
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus
from pixelbox_b200.engine import Engine, IndexedImage
from tests import page_oracle, range_oracle, sqlite_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
INT64_MIN, INT64_MAX = int(np.iinfo(np.int64).min), int(np.iinfo(np.int64).max)


def records(ids, dist, dot, n2):
    return sorted(zip(np.asarray(dist, np.float32).view(np.uint32).tolist(), np.asarray(ids).tolist(), np.asarray(dot).tolist(),
                      np.asarray(n2).tolist()))


def check(got, want, total=None):
    """got: a RangeResult; want: the oracle's (ids, dist, dot, norm2) of the whole answer (or a prefix, total given)."""
    assert list(got.ids) == list(want[0])
    assert np.array_equal(got.dist.view(np.uint32), np.asarray(want[1], np.float32).view(np.uint32))
    # rows that share an image_id and a dist have no defined order among themselves: compare their records as a set
    assert records(got.ids, got.dist, got.dot, got.norm2) == records(*want)
    assert got.total == (len(want[0]) if total is None else total)


def clustered(rng, n, d, spread=3, centres=30):
    cent = rng.integers(0, 256, size=(centres, d))
    return np.clip(cent[rng.integers(0, centres, n)] + rng.integers(-spread, spread + 1, size=(n, d)), 0, 255).astype(np.uint8)


def table(rng, n, d):
    rows = clustered(rng, n, d)
    rows[50:90] = rows[50]                                  # identical rows: ties on dist, broken by image_id
    rows[200:230] = 255 - rows[50]                          # their antipodes: the plateau
    ids = rng.permutation(np.arange(-n // 2, n - n // 2)).astype(np.int64) * 977 + (1 << 33)
    ids[60] = ids[61]                                       # a duplicate image id inside the tie
    ids[0], ids[1] = INT64_MIN + 1, INT64_MAX - 1
    return rows, ids


def radii(dist, rng):
    """From 'exact duplicates only' to 'every row', and the exact dist of rows (that row is out) with the next float up
    (it is in)."""
    s = np.sort(dist)
    picks = [s[min(len(s) - 1, j)] for j in (100, 1000, len(s) // 2)]
    out = [0.0, 1e-3, 0.05, 1e3, 999999.0, 1e7, np.inf, np.nan, -1.0]
    for p in picks:
        out += [float(p), float(np.nextafter(np.float32(p), np.float32(np.inf)))]
    return out


@pytest.mark.parametrize("d", [8, 64, 100, 256, 1024])
def test_range_matches_the_oracle(d):
    rng = np.random.default_rng(d)
    n = 30_000 if d <= 256 else 8_000
    rows, ids = table(rng, n, d)
    qs = [rows[50], rows[7], rng.integers(0, 256, d, dtype=np.uint8)]
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        for q in qs:
            dist = oracle.all_distances(rows, q)
            rs = radii(dist, rng)
            for r in rs:
                want = range_oracle.answer(rows, ids, q, r, dists=dist)
                got = c.search_range(q, r)[0]
                check(got, want)
                assert c.count_within(q, r)[0] == len(want[0])
        # several queries in one call
        counts = c.count_within(np.stack(qs), 0.05)
        assert counts.dtype == np.uint64
        assert counts.tolist() == [len(range_oracle.answer(rows, ids, x, 0.05)[0]) for x in qs]


def test_truncation_paging_and_multi_query_capacity():
    rng = np.random.default_rng(5)
    n, d = 40_000, 64
    rows, ids = table(rng, n, d)
    q = rows[50]
    dist = oracle.all_distances(rows, q)
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        md = float(np.sort(dist)[5000])
        full = range_oracle.answer(rows, ids, q, md, dists=dist)
        total = len(full[0])
        for cap in (1, 7, 100, 2048):
            got = c.search_range(q, md, limit=cap)[0]
            check(got, tuple(a[:cap] for a in full), total)
            top = c.search(q, cap, md)[0]                         # the top-k is the answer's prefix
            assert list(top.ids) == list(got.ids) and np.array_equal(top.dist.view(np.uint32), got.dist.view(np.uint32))
        # chaining `after` reproduces the whole answer
        parts, cur = [], None
        while True:
            g = c.search_range(q, md, limit=997, after=None if cur is None else [cur])[0]
            assert g.total == total - sum(len(p.ids) for p in parts)
            if not len(g.ids):
                break
            parts.append(g)
            cur = (g.dist[-1], int(g.ids[-1]))
        assert list(np.concatenate([p.ids for p in parts])) == list(full[0])
        # one call, three queries, capacity split in query order
        queries = np.stack([rows[50], rows[7], rows[8]])
        wants = [range_oracle.answer(rows, ids, x, md) for x in queries]
        for capacity in (0, 3, len(wants[0][0]) + 5, sum(len(w[0]) for w in wants) + 10):
            hits = np.zeros(max(capacity, 1), nat.HIT_DTYPE)
            off, tot = np.zeros(4, np.uint64), np.zeros(3, np.uint64)
            nat.check(nat.lib().pbx_search_range(c.handle, nat.ptr(queries), 3, md, None, None, 0, nat.PBX_FILTER_EXCLUDE,
                                                 nat.ptr(hits) if capacity else None, capacity, nat.ptr(off), nat.ptr(tot)))
            assert tot.tolist() == [len(w[0]) for w in wants]
            left = capacity
            for i, w in enumerate(wants):
                m = min(left, len(w[0]))
                left -= m
                assert int(off[i + 1] - off[i]) == m
                seg = hits[int(off[i]):int(off[i + 1])]
                assert list(seg["image_id"]) == list(w[0][:m])
                assert np.array_equal(seg["dist"].view(np.uint32), w[1][:m].view(np.uint32))


def test_filters_and_views():
    rng = np.random.default_rng(11)
    n, d = 30_000, 256
    rows, ids = table(rng, n, d)
    fset = ids[rng.random(n) < 0.3]
    allowed = np.isin(ids, fset)
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        with c.view(fset) as v:
            for q in (rows[50], rows[3000]):
                dist = oracle.all_distances(rows, q)
                for md in (0.0, float(np.sort(dist)[3000]), 1e3, 1e7):
                    w_in = range_oracle.answer(rows, ids, q, md, allowed=allowed, dists=dist)
                    w_ex = range_oracle.answer(rows, ids, q, md, allowed=~allowed, dists=dist)
                    check(c.search_range(q, md, within=fset)[0], w_in)
                    check(c.search_range(q, md, excluding=fset)[0], w_ex)
                    check(v.search_range(q, md)[0], w_in)
                    assert c.count_within(q, md, within=fset)[0] == v.count_within(q, md)[0] == len(w_in[0])
                    cur = (w_in[1][len(w_in[1]) // 2], int(w_in[0][len(w_in[0]) // 2])) if len(w_in[0]) else None
                    if cur is not None:
                        w = range_oracle.answer(rows, ids, q, md, cur, allowed, dist)
                        check(v.search_range(q, md, after=[cur])[0], w)
                        check(c.search_range(q, md, within=fset, after=[cur])[0], w)
                        assert c.count_within(q, md, within=fset, after=[cur])[0] == len(w[0])


def test_after_remove_replace_and_pending_appends():
    rng = np.random.default_rng(13)
    n, d = 20_000, 64
    rows, ids = table(rng, n, d)
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids[:n - 100], rows[:n - 100])
        gone = ids[rng.choice(n - 100, 2000, replace=False)]
        c.remove(gone)
        new_rows = clustered(rng, 500, d)
        rep = ids[rng.choice(n - 100, 500, replace=False)]
        rep = rep[~np.isin(rep, gone)]
        c.replace(rep, new_rows[:len(rep)])
        for i in range(n - 100, n):                              # one row per call: coalesced, still pending
            c.append(ids[i:i + 1], rows[i:i + 1])
        t_rows, t_ids = rows.copy(), ids.copy()
        pos = {int(x): i for i, x in enumerate(t_ids)}
        for j, x in enumerate(rep):
            t_rows[pos[int(x)]] = new_rows[j]
        keep = ~np.isin(t_ids, gone)
        t_rows, t_ids = t_rows[keep], t_ids[keep]
        with Corpus(d, capacity_hint=len(t_ids)) as fresh:
            fresh.load(t_ids, t_rows)
            for q in (rows[50], rows[n - 50], new_rows[0]):
                dist = oracle.all_distances(t_rows, q)
                for md in (0.0, float(np.sort(dist)[2000]), 1e7):
                    want = range_oracle.answer(t_rows, t_ids, q, md, dists=dist)
                    check(c.search_range(q, md)[0], want)
                    check(fresh.search_range(q, md)[0], want)


def test_candidate_buffer_regrows():
    # a near-duplicate cluster of 100k rows (more than the first 65536-entry candidate buffer) inside the radius
    rng = np.random.default_rng(17)
    n, d = 150_000, 8
    base = rng.integers(0, 256, d)
    rows = np.concatenate([np.clip(base + rng.integers(-1, 2, size=(100_000, d)), 0, 255),
                           rng.integers(0, 256, size=(n - 100_000, d))]).astype(np.uint8)
    ids = np.arange(n, dtype=np.int64) * 3 - 7
    q = base.astype(np.uint8)
    dist = oracle.all_distances(rows, q)
    md = float(np.sort(dist[:100_000])[-1]) + 1e-3
    want = range_oracle.answer(rows, ids, q, md, dists=dist)
    assert len(want[0]) > 70_000
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        check(c.search_range(q, md)[0], want)
        assert c.count_within(q, md)[0] == len(want[0])
        check(c.search_range(q, md)[0], want)                     # the grown buffer is kept


def test_everything_on_10m_synthetic_rows():
    n, d, seed = 10_000_000, 256, 23
    q = synth.synth_queries(1, 2, d, n, seed)[0]                # a perturbed corpus row
    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed, 0)
        assert c.count_within(q, 1e7)[0] == n
        r = c.search_range(q, 1e7)[0]
        assert r.total == n and len(r.ids) == n
        assert np.array_equal(np.sort(r.ids), np.arange(1, n + 1))   # synthetic ids are row + 1
        key = r.dist.astype(np.float64)
        assert (np.diff(key) >= 0).all()
        same = np.diff(key) == 0
        assert (np.diff(r.ids)[same] > 0).all()                   # ties (the plateau included) by image_id
        rng = np.random.default_rng(1)
        sample = np.concatenate([np.arange(200), rng.choice(n, 2000, replace=False), np.arange(n - 200, n)])
        for i in sample:
            row = synth.synth_rows(seed, int(r.ids[i]) - 1, 1, d)[0]
            assert oracle.cosine_distance(q, row).view(np.uint32) == r.dist[i:i + 1].view(np.uint32)[0]
            assert (int(r.dot[i]), int(r.norm2[i])) == oracle.int_terms(q, row)[::2]
        # the default max_dist (1e3): a count and its answer agree
        t = c.count_within(q, 1e3)[0]
        assert c.search_range(q, 1e3, limit=0)[0].total == t


@pytest.mark.parametrize("devices", [[0, 0, 0], pytest.param([0, 1], marks=pytest.mark.multigpu)])
def test_sharded_equals_one_corpus(devices):
    rng = np.random.default_rng(29)
    n, d = 30_000, 64
    rows, ids = table(rng, n, d)
    rows[n - 20:] = rows[50]                                  # the tie spans the first and the last shard
    fset = ids[::3]
    with MultiDeviceCorpus(d, devices, capacity_hint=n) as m:
        m.load(ids, rows)
        for q in (rows[50], rows[20_000]):
            dist = oracle.all_distances(rows, q)
            for md in (0.0, float(np.sort(dist)[3000]), 1e7):
                want = range_oracle.answer(rows, ids, q, md, dists=dist)
                check(m.search_range(q, md)[0], want)
                assert m.count_within(q, md)[0] == len(want[0])
                for cap in (1, 50, 3001):
                    check(m.search_range(q, md, limit=cap)[0], tuple(a[:cap] for a in want), len(want[0]))
                w = range_oracle.answer(rows, ids, q, md, allowed=np.isin(ids, fset), dists=dist)
                check(m.search_range(q, md, within=fset)[0], w)
                if len(want[0]) > 10:
                    cur = (want[1][5], int(want[0][5]))
                    check(m.search_range(q, md, after=[cur])[0], range_oracle.answer(rows, ids, q, md, cur, dists=dist))


def test_sharded_corpus_world_two():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29657", os.path.join(ROOT, "tools", "range_exchange_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "range_exchange_check OK" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]


def test_range_calls_beside_searches_and_appends():
    rng = np.random.default_rng(31)
    n, d = 50_000, 256
    rows, ids = table(rng, n, d)
    q = rows[50]
    dist = oracle.all_distances(rows, q)
    md = float(np.sort(dist)[4000])
    want = range_oracle.answer(rows, ids, q, md, dists=dist)
    top = page_oracle.page(rows, ids, rows[7], 100, 1e3)
    errors = []
    with Corpus(d, capacity_hint=2 * n) as c:
        c.load(ids, rows)
        stop = threading.Event()

        def searcher():
            while not stop.is_set():
                g = c.search(rows[7], 100, 1e3, within=ids)[0]        # the loaded rows only: appends do not change it
                if list(g.ids) != list(top[0]):
                    errors.append("top-k")

        def appender():
            k = 0
            while not stop.is_set() and k < 200:
                c.append(np.array([(1 << 50) + k], np.int64), rng.integers(0, 256, size=(1, d), dtype=np.uint8))
                k += 1

        th = [threading.Thread(target=searcher), threading.Thread(target=appender)]
        for t in th:
            t.start()
        try:
            for _ in range(20):
                check(c.search_range(q, md, within=ids)[0], want)
                assert c.count_within(q, md, within=ids)[0] == len(want[0])
        finally:
            stop.set()
            for t in th:
                t.join()
    assert not errors


def test_engine_similar_image_ids(tmp_path):
    rng = np.random.default_rng(37)
    n, d = 3000, 64
    rows = clustered(rng, n, d)
    rows[10:30] = rows[10]
    ids = np.arange(1, n + 1, dtype=np.int64)
    db = str(tmp_path / "e.db")
    conn = sqlite_oracle.make_db(db, ids, rows)
    conn.execute("UPDATE images SET path = '/photos/a/' || id || '.png' WHERE id % 2 = 0")
    conn.executemany("DELETE FROM images WHERE id = ?", [(int(i),) for i in ids[15:25]])        # orphan hashes
    conn.commit()
    e = Engine.open(db)
    try:
        img = IndexedImage(visual_hash=bytes(rows[10]))
        for md in (None, 0.0, 0.3):
            got = e.similar_image_ids(img, md)
            sql = conn.execute(sqlite_oracle.similarity_sql(10 ** 9).replace("LIMIT 1000000000", ""),
                               (bytes(rows[10]), float(1e3 if md is None else md))).fetchall()
            assert [g[0] for g in got] == [r[0] for r in sql]
            assert [np.float32(g[1]).view(np.uint32) for g in got] == [np.float32(r[7]).view(np.uint32) for r in sql]
        got = e.similar_image_ids(img, 0.3, folder="/photos/a")
        sql = conn.execute(sqlite_oracle.similarity_sql(10 ** 9).replace("LIMIT 1000000000", "").replace(
            "WHERE dist < ?", "WHERE dist < ? AND substr(images.path, 1, length(?)) = ?"),
            (bytes(rows[10]), 0.3, "/photos/a/", "/photos/a/")).fetchall()
        assert [g[0] for g in got] == [r[0] for r in sql] and len(got) > 0
    finally:
        e.close()
        conn.close()
