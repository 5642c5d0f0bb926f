"""Paged searches (pbx_search_page and its twins, `after=`): every page is the keyset SQL's answer -- the k rows after
the cursor in (dist, image_id) order: ids, dist bit for bit, dot, norm2 and count, compared with the numpy page oracle
(tests/page_oracle.py) -- and the pages of one iteration concatenate to one deep top-K, past PBX_MAX_K."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus, SearchResult
from pixelbox_b200.engine import Engine, IndexedImage
from tests import page_oracle, sqlite_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
INT64_MIN, INT64_MAX = int(np.iinfo(np.int64).min), int(np.iinfo(np.int64).max)


def records(r):
    return sorted(zip(r.dist.view(np.uint32).tolist(), r.ids.tolist(), r.dot.tolist(), r.norm2.tolist()))


def same(a, b):
    """Ids and dist bit for bit in order, and the same (dist, id, dot, norm2) records (rows that share an image_id AND a
    dist have no defined order among themselves), as tests/test_gpu_filter.py compares."""
    return (list(a.ids) == list(b.ids) and np.array_equal(a.dist.view(np.uint32), b.dist.view(np.uint32))
            and records(a) == records(b))


def want(rows, ids, q, k, md, cur=None, allowed=None, dists=None):
    return SearchResult(*page_oracle.page(rows, ids, q, k, md, cur, allowed, dists))


def clustered(rng, n, d, spread=3, centres=30):
    cent = rng.integers(0, 256, size=(centres, d))
    return np.clip(cent[rng.integers(0, centres, n)] + rng.integers(-spread, spread + 1, size=(n, d)), 0, 255).astype(np.uint8)


def last(r):
    return (r.dist[-1], int(r.ids[-1])) if len(r.ids) else None


def iterate(c, rows, ids, queries, k, md, depth, single, allowed=None, within=None, starts=None):
    """Pages of k from `starts` (a cursor or None per query) to `depth` rows; every page is checked against the deep order
    of the oracle.  single: one call per query (the single-query loop), else all queries in one call (batched)."""
    nq = len(queries)
    dists = [page_oracle.order(rows, ids, q, md, allowed) for q in queries]
    curs = list(starts) if starts is not None else [None] * nq
    pos = [len(full) - len(page_oracle.after_cursor(full, ids, dist, cur)) for (full, dist), cur in zip(dists, curs)]
    done = [False] * nq
    for _ in range(0, depth, k):
        if single:
            got = [c.search(queries[i], k, md, after=[curs[i]], within=within)[0] for i in range(nq)]
        else:
            got = c.search(queries, k, md, after=curs, within=within)
        for i, g in enumerate(got):
            full, dist = dists[i]
            sel = full[pos[i]:pos[i] + k]
            w = SearchResult(ids[sel], dist[sel], *page_oracle.centred_terms(rows[sel], queries[i]))
            assert same(g, w), f"k={k} md={md} query {i} at depth {pos[i]} single={single}"
            pos[i] += len(g.ids)
            if len(g.ids):
                curs[i] = last(g)
            done[i] = len(g.ids) < k
        if all(done):
            break
    return pos


# ---- deep iteration: page sizes, dims, max_dist, both paths, mixed cursors, forced exact pass ------------------------
@pytest.mark.parametrize("d", [8, 100, 256, 1024])
def test_pages_concatenate_to_one_deep_top_k(d):
    rng = np.random.default_rng(500 + d)
    n = 12_000
    rows = clustered(rng, n, d)
    rows[100:160] = rows[100]                               # a tie of identical rows
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 5
    queries = np.concatenate([rows[[100, 4000]], rng.integers(0, 256, size=(2, d), dtype=np.uint8)])
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        b0 = c.stats().batched_queries
        c.search(queries, 100)
        batched = c.stats().batched_queries > b0           # whether this shape has a tensor-core path at all
        for slack in (0, 1):
            c.set_candidate_slack(slack)
            xp0 = c.stats().exact_passes
            for md in (1e3, 0.05, 1e7):
                for k, depth in ((100, 10_000), (2048, 10_000), (7, 700), (1, 60)):
                    if slack == 1 and k in (1, 2048) and d != 256:
                        continue
                    iterate(c, rows, ids, queries[:2], k, md, depth, single=True)
                    if k <= 1000:
                        # batched: the first page (NULL), -inf, and a cursor at another depth for every query
                        full, dist = page_oracle.order(rows, ids, queries[2], md)
                        mid = (dist[full[min(333, len(full) - 1)]], int(ids[full[min(333, len(full) - 1)]])) if len(full) else None
                        starts = [None, (np.float32(-np.inf), INT64_MIN), mid, None]
                        b0 = c.stats().batched_queries
                        iterate(c, rows, ids, queries, k, md, depth, single=False, starts=starts)
                        if slack == 0:
                            assert (c.stats().batched_queries > b0) == batched, "the paged batch took another path"
            if slack == 1:
                assert c.stats().exact_passes > xp0, "a candidate slack of 1 forced no exact pass"


# ---- cursor edges ------------------------------------------------------------------------------------------------------
def test_cursor_edges():
    rng = np.random.default_rng(7)
    d, n = 64, 20_000
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    rows[1000:1700] = rows[1000]                           # a 700-row tie of identical rows
    ids = rng.permutation(np.arange(-n // 2, n - n // 2)).astype(np.int64) * 3 + 1
    ids[1000], ids[1001], ids[1002] = INT64_MIN, INT64_MAX, 0
    ids[5000:5003] = ids[4999]                             # one id on several rows
    q_tie = rows[1000]
    q_anti = (255 - rows[7]).astype(np.uint8)              # its plateau holds most rows
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        for q in (q_tie, q_anti, rows[5000]):
            dist = page_oracle.order(rows, ids, q, 1e7)[1]
            tie_d = dist[1000]
            step = np.nextafter(np.float32(0.3), np.float32(1))
            curs = [(tie_d, INT64_MIN), (tie_d, 0), (tie_d, int(ids[1500])), (tie_d, INT64_MAX),
                    (np.float32(-1.1920929e-07), INT64_MIN), (np.float32(-1.1920929e-07), 0),
                    (np.float32(-1.0), 0), (np.float32(-0.5), 5), (np.float32(0.0), 0), (np.float32(np.inf), INT64_MIN),
                    (np.float32(-np.inf), INT64_MIN), (np.float32(-np.inf), INT64_MAX),
                    (np.float32(999999.0), INT64_MIN), (np.float32(999999.0), int(ids[9000])), (np.float32(2e6), 0),
                    (np.float32(0.3), 2), (step, 2), (np.float32(0.7123), 424242),       # no row
                    (dist[5000], int(ids[5000])), (dist[5000], int(ids[5000]) - 1)]          # duplicate ids
            srt = np.unique(dist)
            for j in (5, len(srt) // 2):                                                    # one ulp either side of a dist step
                curs += [(srt[j], INT64_MAX), (np.nextafter(srt[j], np.float32(-1)), INT64_MAX),
                         (np.nextafter(srt[j], np.float32(2)), INT64_MIN)]
            for md in (1e3, 1e7):
                for k in (1, 100, 700):
                    for cur in curs:
                        w = want(rows, ids, q, k, md, cur, dists=dist)
                        assert same(c.search(q, k, md, after=[cur])[0], w), f"single k={k} md={md} cursor {cur}"
                    got = c.search(np.stack([q] * len(curs)), k, md, after=curs)
                    for cur, g in zip(curs, got):
                        assert same(g, want(rows, ids, q, k, md, cur, dists=dist)), f"batched k={k} md={md} cursor {cur}"
        # the id of a removed row
        gone = int(ids[3000])
        c.remove([gone])
        keep = ids != gone
        q = rows[3000]
        dist = page_oracle.order(rows[keep], ids[keep], q, 1e3)[1]
        d_gone = page_oracle.order(rows[3000:3001], ids[3000:3001], q, 1e3)[1][0]
        for cur in ((d_gone, gone), (d_gone, gone - 1), (d_gone, gone + 1)):
            assert same(c.search(q, 100, 1e3, after=[cur])[0], want(rows[keep], ids[keep], q, 100, 1e3, cur, dists=dist))


def test_nan_cursor():
    rng = np.random.default_rng(9)
    rows = rng.integers(0, 256, size=(5000, 32), dtype=np.uint8)
    ids = np.arange(5000, dtype=np.int64)
    with Corpus(32, capacity_hint=5000) as c:
        c.load(ids, rows)
        with pytest.raises(nat.PbxError):
            c.search(rows[0], 10, after=[(np.nan, 1)])
        # the device form: count 0 for that query only
        cur = np.zeros(2, nat.HIT_DTYPE)
        cur["dist"] = [np.nan, -np.inf]
        cur["image_id"] = [1, INT64_MIN]
        d_q = torch.from_numpy(rows[:2].copy()).cuda()
        d_after = torch.from_numpy(cur.view(np.uint8).copy()).cuda()
        d_hits = torch.zeros(2 * 10 * 24, dtype=torch.uint8, device="cuda")
        d_cnt = torch.zeros(2, dtype=torch.int32, device="cuda")
        c.search_device_page(d_q.data_ptr(), 2, 10, 1e3, d_hits.data_ptr(), d_cnt.data_ptr(), d_after.data_ptr())
        c.synchronize()
        assert d_cnt.cpu().tolist() == [0, 10]


# ---- every rank of a clustered corpus as a cursor --------------------------------------------------------------------
def test_every_rank_as_a_cursor():
    rng = np.random.default_rng(11)
    d, n = 64, 3000
    rows = clustered(rng, n, d, spread=2, centres=5)
    ids = rng.permutation(n).astype(np.int64)
    q = rows[17]
    full, dist = page_oracle.order(rows, ids, q, 1e3)
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        for r in range(len(full)):
            cur = (dist[full[r]], int(ids[full[r]]))
            sel = full[r + 1:r + 11]
            w = SearchResult(ids[sel], dist[sel], *page_oracle.centred_terms(rows[sel], q))
            assert same(c.search(q, 10, 1e3, after=[cur])[0], w), f"rank {r}"


# ---- filters, remove, pending appends ----------------------------------------------------------------------------------
def test_pages_with_filters_remove_and_appends():
    rng = np.random.default_rng(13)
    d, n = 96, 30_000
    rows = clustered(rng, n, d)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    queries = rows[[3, 12_000]]
    with Corpus(d, capacity_hint=2 * n) as c:
        c.load(ids, rows)
        for name, fset in (("dense", ids[rng.random(n) < 0.5]), ("1%", ids[rng.random(n) < 0.01])):
            for kw in ("within", "excluding"):
                allowed = np.isin(ids, fset) if kw == "within" else ~np.isin(ids, fset)
                for single in (True, False):
                    curs = [None, None]
                    for _ in range(12):
                        got = ([c.search(queries[i], 100, 1e3, after=[curs[i]], **{kw: fset})[0] for i in range(2)] if single
                               else c.search(queries, 100, 1e3, after=curs, **{kw: fset}))
                        for i, g in enumerate(got):
                            assert same(g, want(rows, ids, queries[i], 100, 1e3, curs[i], allowed)), f"{name} {kw} single={single}"
                            curs[i] = last(g) or curs[i]
        # remove a third, then append rows that sort before and after a cursor (pending: searches flush them)
        cur = last(c.search(queries[0], 500, 1e3)[0])
        gone = ids[::3]
        c.remove(gone)
        live = ~np.isin(ids, gone)
        new_rows = np.concatenate([rows[[3] * 4], rows[rng.integers(0, n, 200)]])
        new_ids = np.arange(n + 1, n + 1 + len(new_rows), dtype=np.int64)
        c.append(new_ids, new_rows)
        all_rows, all_ids = np.concatenate([rows[live], new_rows]), np.concatenate([ids[live], new_ids])
        for single in (True, False):
            got = c.search(queries[0], 300, 1e3, after=[cur])[0] if single else c.search(queries, 300, 1e3, after=[cur, None])[0]
            assert same(got, want(all_rows, all_ids, queries[0], 300, 1e3, cur))


# ---- the device form chains pages without a host read -------------------------------------------------------------------
def test_device_form_chains_pages():
    rng = np.random.default_rng(17)
    d, n, k, nq = 128, 50_000, 100, 3
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = np.arange(n, dtype=np.int64) * 2
    queries = rows[[1, 2, 3]]
    fset = ids[rng.random(n) < 0.3]
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        d_q = torch.from_numpy(queries.copy()).cuda()
        d_f = torch.from_numpy(np.sort(fset)).cuda()
        for filt in (False, True):
            for q_at_once in (1, nq):
                pages = 6
                d_hits = [torch.zeros(q_at_once * k * 24, dtype=torch.uint8, device="cuda") for _ in range(pages)]
                d_cnt = [torch.zeros(q_at_once, dtype=torch.int32, device="cuda") for _ in range(pages)]
                d_curs = []
                s = torch.cuda.current_stream()
                for p in range(pages):
                    after = 0
                    if p:
                        # each query's cursor is the record at slot k - 1 of its previous page (pages here are full),
                        # gathered on the stream: no host read
                        d_curs.append(d_hits[p - 1].view(q_at_once, k, 24)[:, k - 1, :].contiguous())
                        after = d_curs[-1].data_ptr()
                    c.search_device_page(d_q.data_ptr(), q_at_once, k, 1e3, d_hits[p].data_ptr(), d_cnt[p].data_ptr(), after,
                                         d_f.data_ptr() if filt else 0, d_f.numel() if filt else 0,
                                         nat.PBX_FILTER_INCLUDE if filt else nat.PBX_FILTER_EXCLUDE, s.cuda_stream)
                torch.cuda.synchronize()
                allowed = np.isin(ids, fset) if filt else None
                for i in range(q_at_once):
                    full, dist = page_oracle.order(rows, ids, queries[i], 1e3, allowed)
                    for p in range(pages):
                        h = d_hits[p].cpu().numpy().view(nat.HIT_DTYPE).reshape(q_at_once, k)[i]
                        assert int(d_cnt[p][i]) == k
                        got = SearchResult(h["image_id"].copy(), h["dist"].copy(), h["dot"].copy(), h["norm2"].copy())
                        sel = full[p * k:(p + 1) * k]
                        assert same(got, SearchResult(ids[sel], dist[sel], *page_oracle.centred_terms(rows[sel], queries[i])))


# ---- sharding ------------------------------------------------------------------------------------------------------------
def test_three_shards_on_one_device():
    rng = np.random.default_rng(19)
    d, n = 64, 30_000
    rows = clustered(rng, n, d)
    ids = rng.permutation(n).astype(np.int64)
    queries = rows[[0, 9]]
    with MultiDeviceCorpus(d, [0, 0, 0], capacity_hint=n) as s:
        s.load(ids, rows)
        fset = ids[::2]
        for kw, allowed in ((None, None), ("within", np.isin(ids, fset))):
            extra = {} if kw is None else {kw: fset}
            curs = [None, (np.float32(-np.inf), INT64_MIN)]
            for _ in range(8):
                got = s.search(queries, 250, 1e3, after=curs, **extra)
                for i, g in enumerate(got):
                    assert same(g, want(rows, ids, queries[i], 250, 1e3, curs[i], allowed))
                    curs[i] = last(g) or curs[i]


def test_sharded_corpus_between_processes_sharing_one_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29702", os.path.join(ROOT, "tools", "page_exchange_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "page_exchange_check OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


# ---- the band: exclusions beyond the slack, and the above-cut count ----------------------------------------------------
def test_cursor_inside_a_cluster_larger_than_the_batched_buffers():
    rng = np.random.default_rng(23)
    d, n_other, n_cluster = 128, 40_000, 9000
    base = rng.integers(0, 256, size=d)
    cluster = np.clip(base + rng.integers(-1, 2, size=(n_cluster, d)), 0, 255).astype(np.uint8)
    rows = np.concatenate([rng.integers(0, 256, size=(n_other, d), dtype=np.uint8), cluster])
    ids = rng.permutation(len(rows)).astype(np.int64)
    q = base.astype(np.uint8)
    full, dist = page_oracle.order(rows, ids, q, 1e3)
    with Corpus(d, capacity_hint=len(rows)) as c:
        c.load(ids, rows)
        for r in (4000, 8500):                            # inside the cluster: the band holds most candidates
            cur = (dist[full[r]], int(ids[full[r]]))
            xp0 = c.stats().exact_passes
            assert same(c.search(q, 100, 1e3, after=[cur])[0], want(rows, ids, q, 100, 1e3, cur, dists=dist))
            got = c.search(np.stack([q] * 4), 100, 1e3, after=[cur] * 4)
            assert all(same(g, want(rows, ids, q, 100, 1e3, cur, dists=dist)) for g in got)
            assert c.stats().exact_passes > xp0, "the band left fewer than k candidates, yet no exact pass ran"


def test_paging_to_exhaustion_needs_no_exact_pass():
    rng = np.random.default_rng(29)
    d, n = 64, 5000
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = rng.permutation(n).astype(np.int64)
    queries = rows[[1, 2]]
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        for single in (True, False):
            xp0 = c.stats().exact_passes
            pos = iterate(c, rows, ids, queries, 100, 1e3, n + 100, single=single)
            assert all(p == len(page_oracle.order(rows, ids, q, 1e3)[0]) for p, q in zip(pos, queries))
            assert c.stats().exact_passes == xp0, f"paging to exhaustion took exact passes (single={single})"


# ---- Engine ------------------------------------------------------------------------------------------------------------
def engine_db(tmp_path, n_orphans, n_images, d=64, seed=31):
    rng = np.random.default_rng(seed)
    q = rng.integers(0, 256, size=d, dtype=np.uint8)
    near = np.clip(q.astype(int) + rng.integers(-2, 3, size=(n_orphans, d)), 0, 255).astype(np.uint8)
    far = rng.integers(0, 256, size=(n_images, d), dtype=np.uint8)
    hashes = np.concatenate([near, far])
    ids = np.arange(1, len(hashes) + 1, dtype=np.int64)
    path = str(tmp_path / "engine.db")
    conn = sqlite_oracle.make_db(path, ids, hashes)
    # the nearest hashes lose their images row (an external tool deleted a folder's images)
    conn.execute(f"DELETE FROM images WHERE id <= {n_orphans}")
    conn.execute("UPDATE images SET path = '/f/' || filename WHERE id % 2 = 0")
    conn.commit()
    return path, conn, q


def sql_rows(conn, q, md, limit, offset=0, folder=None):
    sql = sqlite_oracle.similarity_sql(limit + offset)
    if folder is not None:
        sql = sql.replace("WHERE dist < ?", "WHERE dist < ? AND substr(images.path, 1, length(?)) = ?")
        rows = conn.execute(sql, (bytes(q), float(md), folder, folder)).fetchall()
    else:
        rows = conn.execute(sql, (bytes(q), float(md))).fetchall()
    return [(r[0], np.float32(r[7])) for r in rows][offset:]


def test_engine_orphan_hashes_and_load_more(tmp_path):
    path, conn, q = engine_db(tmp_path, 2500, 3000)
    eng = Engine.open(path)
    try:
        img = IndexedImage(visual_hash=bytes(q))
        eng.query_by_image_hash_from_image(img)
        got = [(r.id, np.float32(r.distance_from_query)) for r in eng.get_query_results()]
        assert len(got) == 100 and got == sql_rows(conn, q, 1e3, 100)
        for p in range(1, 4):
            eng.load_more_results()
            got = [(r.id, np.float32(r.distance_from_query)) for r in eng.get_query_results()]
            assert got[100 * p:] == sql_rows(conn, q, 1e3, 100, 100 * p), f"page {p}"
        eng.query_by_image_hash_within_folder(img, "/f")
        assert [(r.id, np.float32(r.distance_from_query)) for r in eng.get_query_results()] == sql_rows(conn, q, 1e3, 100, folder="/f/")
        for p in range(1, 3):
            eng.load_more_results()
            got = [(r.id, np.float32(r.distance_from_query)) for r in eng.get_query_results()]
            assert got[100 * p:] == sql_rows(conn, q, 1e3, 100, 100 * p, folder="/f/"), f"folder page {p}"
        # the end of the table: load_more stops adding rows
        eng.max_distance_from_query = 0.02
        eng.query_by_image_hash_from_image(img)
        first = eng.get_query_results()
        eng.load_more_results()
        assert eng.get_query_results() == first
    finally:
        eng.close()
        conn.close()
