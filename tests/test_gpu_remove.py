"""pbx_corpus_remove / pbx_sharded_remove: after a removal every search path returns exactly what a corpus loaded with
the surviving rows returns (ids, dist bit for bit, dot, norm2), the layout follows the hole-filling rule, rows left
behind past the end are never read, and removal is ordered against searches already enqueued."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def test_remove_argument_errors_need_no_gpu():
    L = nat.lib()
    ids = np.array([1, 2], np.int64)
    out = ctypes.c_uint64(7)
    assert L.pbx_corpus_remove(None, nat.ptr(ids), 2, ctypes.byref(out)) == -1 and out.value == 0
    assert L.pbx_corpus_remove(None, None, 2, None) == -1
    assert L.pbx_sharded_remove(None, nat.ptr(ids), 2, None) == -1
    assert L.pbx_sharded_remove(None, None, 1, ctypes.byref(out)) == -1


# ---- helpers ------------------------------------------------------------------------------------------------------------
def same(res, want):
    o_ids, o_dist, o_dot, o_n2 = want
    return (list(res.ids) == list(o_ids) and np.array_equal(res.dist.view(np.uint32), np.asarray(o_dist).view(np.uint32))
            and np.array_equal(res.dot, o_dot) and np.array_equal(res.norm2, o_n2))


def same_res(a, b):
    return same(a, (b.ids, b.dist, b.dot, b.norm2))


def hole_fill(ids, rows, gone):
    """The documented layout: the j-th removed row below n' receives the j-th surviving row at or above n'."""
    nk = len(ids) - int(gone.sum())
    out_ids, out_rows = ids[:nk].copy(), rows[:nk].copy()
    holes = np.flatnonzero(gone[:nk])
    srcs = nk + np.flatnonzero(~gone[nk:])
    assert len(holes) == len(srcs)
    out_ids[holes], out_rows[holes] = ids[srcs], rows[srcs]
    return out_ids, out_rows


def clustered(rng, n, d, spread=3, centres=30):
    cent = rng.integers(0, 256, size=(centres, d))
    return np.clip(cent[rng.integers(0, centres, n)] + rng.integers(-spread, spread + 1, size=(n, d)), 0, 255).astype(np.uint8)


def check_layout(c, ids, rows, gone):
    want_ids, want_rows = hole_fill(ids, rows, gone)
    got_ids, got_rows = c.read_rows(0, len(want_ids))
    assert np.array_equal(got_ids, want_ids) and np.array_equal(got_rows, want_rows)
    assert len(c) == len(want_ids) and c.stats().rows == len(want_ids)
    return want_ids, want_rows


# ---- single-query path: every kind of removal, every k / max_dist, with and without the exact pass ------------------------
@gpu
@pytest.mark.parametrize("d", [8, 100, 256])
def test_single_query_parity_after_removal(d):
    rng = np.random.default_rng(700 + d)
    n = 12_000
    rows = clustered(rng, n, d)
    rows[50:80] = rows[50]                        # a duplicated hash at the front ...
    rows[n - 20:] = rows[50]                      # ... and in the tail
    ids = (rng.permutation(np.arange(1, n + 1)) * 3).astype(np.int64)
    nk_run = n - 200
    sets = {
        "nothing": np.array([-5, 2, 10**12], np.int64),                        # ids are multiples of 3
        "one": ids[[1234]],
        "first": ids[:100],
        "tail": ids[n - 50:],
        "straddle": ids[nk_run - 100:nk_run + 100],
        "random10": ids[rng.random(n) < 0.10],
        "dup_all": np.concatenate([ids[50:80], ids[n - 20:]]),
        "dup_half": ids[50:65],
    }
    for name, req in sets.items():
        gone = np.isin(ids, req)
        with Corpus(d, capacity_hint=n) as c:
            c.load(ids, rows)
            cap = c.stats().capacity_rows
            assert c.remove(np.concatenate([req, req[:3]])) == int(gone.sum()), name      # repeats count once
            assert c.stats().capacity_rows == cap
            s_ids, s_rows = check_layout(c, ids, rows, gone)
            removed = set(ids[gone].tolist())
            qi = np.flatnonzero(gone)[:2].tolist() + [50, int(np.flatnonzero(~gone)[0])]
            queries = np.concatenate([rows[qi], rng.integers(0, 256, size=(1, d), dtype=np.uint8)])
            for slack in (0, 1):
                c.set_candidate_slack(slack)
                for k in (10, 100, 1000):
                    for md in (1e3, 0.05, 1e7):
                        for j, q in enumerate(queries):
                            got = c.search(q, k, md)[0]
                            want = oracle.topk(s_rows, s_ids, q, k, md, threads=4)
                            assert same(got, want), f"{name} d={d} slack={slack} k={k} md={md} q={j}"
                            assert not removed.intersection(got.ids.tolist())


# ---- rows past the new end are stale and must never be read ---------------------------------------------------------------
@gpu
def test_stale_tail_is_never_read():
    rng = np.random.default_rng(5)
    n, d = 50_000, 64
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = np.arange(1, n + 1, dtype=np.int64)
    with Corpus(d) as c:
        c.load(ids, rows)
        gone = np.zeros(n, bool)
        gone[:10] = True
        gone[n - 3] = True                        # a removed row in the tail region
        assert c.remove(ids[gone]) == 11
        check_layout(c, ids, rows, gone)
        moved = n - 1                             # a survivor at or above n' = n - 11: it moved into a hole
        before = c.stats().batched_queries
        queries = np.concatenate([rows[[moved, n - 3]], rng.integers(0, 256, size=(30, d), dtype=np.uint8)])
        for res in (c.search(queries[:1], 100, 1e7), c.search(queries[1:2], 100, 1e7), c.search(queries, 100, 1e7)):
            for r in res:
                assert list(r.ids).count(ids[moved]) <= 1 and ids[n - 3] not in r.ids.tolist()
        for r in (c.search(queries[:1], 100, 1e7)[0], c.search(queries, 100, 1e7)[0]):
            assert r.ids[0] == ids[moved] and list(r.ids).count(ids[moved]) == 1
        assert c.stats().batched_queries > before


# ---- tensor-core batched path -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", [64, 256])
def test_batched_path_after_removing_30_percent(d):
    rng = np.random.default_rng(900 + d)
    n = 200_000
    rows = clustered(rng, n, d, spread=4, centres=200)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    gone = rng.random(n) < 0.30
    with Corpus(d) as c:
        c.load(ids, rows)
        assert c.remove(ids[gone]) == int(gone.sum())
        s_ids, s_rows = check_layout(c, ids, rows, gone)
        queries = np.concatenate([rows[np.flatnonzero(gone)[:64]], rows[np.flatnonzero(~gone)[:64]],
                                  rng.integers(0, 256, size=(128, d), dtype=np.uint8)])
        for k, md in ((100, 1e3), (10, 0.05)):
            before = c.stats().batched_queries
            got = c.search(queries, k, md)
            assert c.stats().batched_queries == before + len(queries)
            c.set_batch_min(0xFFFFFFFF)
            ref = c.search(queries, k, md)
            c.set_batch_min(0)
            for i in range(len(queries)):
                assert same_res(got[i], ref[i]), (k, md, i)
            for i in list(range(0, len(queries), 37)) + [0, 64]:
                assert same(got[i], oracle.topk(s_rows, s_ids, queries[i], k, md, threads=8)), (k, md, i)


@gpu
def test_moved_row_with_extreme_norm_is_found_by_the_batched_path():
    """A row with a norm / row term far outside the bounds of the block it moves into: the block metadata must be
    recomputed or the batched epilogue's one-compare test rejects it.  The front rows are low bytes (norms near the
    largest, row terms near the smallest); the planted row alternates 127 / 128 (norm^2 = d, row term 0).  Queried with
    its own bytes it is the only good match (cosine 1, every other row ~0.01), but its dot product is tiny: against
    the stale block bounds (large minimum norm, very negative row term) it cannot reach the threshold."""
    rng = np.random.default_rng(17)
    n, d = 60_000, 64
    rows = rng.integers(0, 16, size=(n, d), dtype=np.uint8)                # near-uniform front, low bytes
    rows[n - 1] = np.where(np.arange(d) % 2 == 0, 127, 128)                # smallest norm, row term 0
    rows[n - 2] = 255                                                      # largest norm and row term
    ids = np.arange(1, n + 1, dtype=np.int64)
    with Corpus(d) as c:
        c.load(ids, rows)
        gone = np.zeros(n, bool)
        gone[[3, 40]] = True                      # blocks 0 and 1 receive the two planted rows
        assert c.remove(ids[gone]) == 2
        s_ids, s_rows = check_layout(c, ids, rows, gone)
        assert set(s_ids[[3, 40]].tolist()) == {n, n - 1}
        queries = np.concatenate([rows[[n - 1, n - 2]], rng.integers(0, 256, size=(30, d), dtype=np.uint8)])
        before = c.stats().batched_queries
        got = c.search(queries, 10, 1e3)
        assert c.stats().batched_queries == before + len(queries)
        assert got[0].ids[0] == n and got[0].dist[0] <= 1e-6 and got[1].ids[0] == n - 1
        for i in range(4):
            assert same(got[i], oracle.topk(s_rows, s_ids, queries[i], 10, 1e3, threads=8)), i


# ---- edge cases ---------------------------------------------------------------------------------------------------------
@gpu
def test_remove_edge_cases():
    rng = np.random.default_rng(3)
    d = 32
    rows = rng.integers(0, 256, size=(3000, d), dtype=np.uint8)
    ids = np.arange(1, 3001, dtype=np.int64)
    L = nat.lib()
    # room for the appends below and the append path's growth head-room (4096 rows ahead): capacity must not change
    with Corpus(d, capacity_hint=16384) as c:
        out = ctypes.c_uint64(9)
        assert c.remove([1, 2]) == 0                                          # empty corpus
        assert L.pbx_corpus_remove(c.handle, None, 1, None) == -1
        assert L.pbx_corpus_remove(c.handle, None, 0, ctypes.byref(out)) == 0 and out.value == 0
        c.load(ids, rows)
        cap = c.stats().capacity_rows
        # pending (coalesced) appends are subject to the removal
        c.append([5000, 5001], rows[:2])
        assert len(c) == 3002
        assert c.remove([5001, 7]) == 2 and len(c) == 3000
        got = c.search(rows[0], 5, 1e7)[0]
        assert list(got.ids[:2]) == [1, 5000]
        assert 5001 not in c.search(rows[1], 5, 1e7)[0].ids
        # duplicate ids in the corpus: every row goes
        c.append(np.full(100, 4242, np.int64), rows[:100])
        assert c.remove(np.array([4242, 4242, 4242], np.int64)) == 100
        assert 4242 not in c.search(rows[0], 10, 1e7)[0].ids
        # remove, then append the same id with new bytes: a replace
        new = rng.integers(0, 256, size=(1, d), dtype=np.uint8)
        assert c.remove([10]) == 1
        c.append([10], new)
        r = c.search(new[0], 1, 1e7)[0]
        assert list(r.ids) == [10] and r.dist[0] <= 1e-6
        r2 = c.search(rows[9], 3, 1e7)[0]
        assert r2.ids[0] != 10 or r2.dist[0] > 0.0
        assert c.stats().capacity_rows == cap                                # appends reused the freed rows
        # remove everything, then start again
        all_ids, _ = c.read_rows(0, len(c))
        assert c.remove(all_ids) == len(all_ids) and len(c) == 0
        assert c.search(rows[0], 10, 1e7)[0].ids.size == 0
        assert c.search(rows[:4], 10, 1e7)[3].ids.size == 0
        c.append([77], rows[5:6])
        assert list(c.search(rows[5], 10, 1e7)[0].ids) == [77]
        assert c.stats().capacity_rows == cap


# ---- ordering against device searches already enqueued ---------------------------------------------------------------
@gpu
def test_removal_waits_for_enqueued_device_searches():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(11)
    n, d, k, nq = 400_000, 256, 100, 64
    rows = clustered(rng, n, d, spread=4, centres=300)
    ids = np.arange(1, n + 1, dtype=np.int64)
    queries = rows[rng.integers(0, n, 8 * nq)]
    gone = rng.random(n) < 0.2
    with Corpus(d, device=0) as c:
        c.load(ids, rows)
        before = c.search(queries, k, 1e3)
        dev = torch.device("cuda", 0)
        stream = torch.cuda.Stream(dev)
        dq = torch.from_numpy(queries).to(dev)
        torch.cuda.synchronize(dev)
        hits = [torch.empty(nq * k * nat.HIT_DTYPE.itemsize, dtype=torch.uint8, device=dev) for _ in range(8)]
        cnts = [torch.empty(nq, dtype=torch.int32, device=dev) for _ in range(8)]
        for i in range(8):
            c.search_device(dq[i * nq:(i + 1) * nq].data_ptr(), nq, k, 1e3, hits[i].data_ptr(), cnts[i].data_ptr(), stream.cuda_stream)
        assert c.remove(ids[gone]) == int(gone.sum())                        # no synchronisation before this
        h_after = torch.empty(nq * k * nat.HIT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        c_after = torch.empty(nq, dtype=torch.int32, device=dev)
        c.search_device(dq[:nq].data_ptr(), nq, k, 1e3, h_after.data_ptr(), c_after.data_ptr(), stream.cuda_stream)
        stream.synchronize()
        for i in range(8):
            h = hits[i].cpu().numpy().view(nat.HIT_DTYPE).reshape(nq, k)
            cnt = cnts[i].cpu().numpy()
            for j in range(nq):
                b = before[i * nq + j]
                assert cnt[j] == len(b.ids) and list(h[j]["image_id"][:cnt[j]]) == list(b.ids), (i, j)
                assert np.array_equal(h[j]["dist"][:cnt[j]].view(np.uint32), b.dist.view(np.uint32))
        after = c.search(queries[:nq], k, 1e3)
        h = h_after.cpu().numpy().view(nat.HIT_DTYPE).reshape(nq, k)
        cnt = c_after.cpu().numpy()
        removed = set(ids[gone].tolist())
        for j in range(nq):
            assert cnt[j] == len(after[j].ids) and list(h[j]["image_id"][:cnt[j]]) == list(after[j].ids), j
            assert np.array_equal(h[j]["dist"][:cnt[j]].view(np.uint32), after[j].dist.view(np.uint32))
            assert not removed.intersection(after[j].ids.tolist())


# ---- scale ---------------------------------------------------------------------------------------------------------------
@gpu
def test_remove_at_scale_equals_a_reloaded_corpus():
    from pixelbox_b200 import synth
    n, d = 2_000_000, 256
    rng = np.random.default_rng(29)
    with Corpus(d, capacity_hint=n + 64) as c:
        c.fill_synthetic(n, 42)
        dup_src = rng.choice(n, 8, replace=False)
        _, dup_rows = c.read_rows(int(dup_src[0]), 1)
        planted = np.stack([synth.synth_rows(42, int(r), 1, d)[0] for r in dup_src])
        assert np.array_equal(planted[0], dup_rows[0])
        c.append(np.repeat(dup_src + 1, 3).astype(np.int64), np.repeat(planted, 3, axis=0))      # each id on four rows
        gone_ids = np.unique(np.concatenate([rng.choice(np.arange(1, n + 1), n // 100, replace=False), dup_src + 1])).astype(np.int64)
        assert c.remove(gone_ids) == len(gone_ids) + 3 * len(dup_src)
        nk = len(c)
        assert nk == n + 3 * len(dup_src) - (len(gone_ids) + 3 * len(dup_src))
        s_ids, s_rows = c.read_rows(0, nk)
        assert not np.isin(s_ids, gone_ids).any()
        with Corpus(d, capacity_hint=nk) as fresh:
            fresh.load(s_ids, s_rows)
            queries = np.concatenate([planted[:4], synth.synth_queries(7, 1024, d, n, 42)])
            removed = set(gone_ids.tolist())
            for q in queries[:64]:
                a, b = c.search(q, 100, 1e3)[0], fresh.search(q, 100, 1e3)[0]
                assert same_res(a, b) and not removed.intersection(a.ids.tolist())
            a, b = c.search(queries[:1024], 100, 1e3), fresh.search(queries[:1024], 100, 1e3)
            for i in range(1024):
                assert same_res(a[i], b[i]) and not removed.intersection(a[i].ids.tolist()), i


# ---- several devices, one process -----------------------------------------------------------------------------------------
def devices(n):
    have = max(1, nat.lib().pbx_device_count())
    return [i % have for i in range(n)]


@gpu
def test_multi_device_corpus_remove():
    rng = np.random.default_rng(41)
    n, d = 60_000, 256
    rows = clustered(rng, n, d, spread=2, centres=40)
    rows[100:300] = rows[100]
    rows[n - 300:] = rows[100]                    # a plateau in the first and in the last shard
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 3
    gone = rng.random(n) < 0.05
    gone[150:250] = True                          # part of the tie in shard 0 ...
    gone[n - 100:] = True                         # ... and in shard 2
    queries = np.concatenate([rows[[100, 20_000, 45_000]], rng.integers(0, 256, size=(20, d), dtype=np.uint8)])
    with MultiDeviceCorpus(d, devices(3)) as mc:
        mc.load(ids, rows)
        removed = mc.remove(ids[gone])
        assert removed == int(gone.sum()) and len(mc) == n - removed
        s_ids, s_rows = ids[~gone], rows[~gone]
        for k, md, qs in ((100, 1e3, queries), (300, 1e7, queries[:2]), (10, 0.02, queries[:3])):
            got = mc.search(qs, k, md)
            for qi, q in enumerate(qs):
                assert same(got[qi], oracle.topk(s_rows, s_ids, q, k, md, threads=8)), (k, md, qi)
        sizes = [mc.shard_stats(i).rows for i in range(3)]
        mc.append([10**9], queries[3:4])
        after = [mc.shard_stats(i).rows for i in range(3)]
        smallest = int(np.argmin(sizes))
        assert after[smallest] == sizes[smallest] + 1 and sum(after) == sum(sizes) + 1
        assert mc.search(queries[3], 1, 1e3)[0].ids[0] == 10**9


# ---- one process per rank -----------------------------------------------------------------------------------------------
@gpu
def test_sharded_corpus_remove_between_processes_sharing_one_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29671", os.path.join(ROOT, "tools", "remove_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "remove_check OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


# ---- the Engine mirror ---------------------------------------------------------------------------------------------------
@gpu
def test_engine_remove_images_matches_verbatim_sql(tmp_path):
    from pixelbox_b200.engine import Engine, IndexedImage
    from tests import sqlite_oracle
    rng = np.random.default_rng(8)
    n, d = 4000, 64
    rows = clustered(rng, n, d)
    rows[10:70] = rows[10]
    ids = np.arange(1, n + 1, dtype=np.int64)
    path = str(tmp_path / "remove.db")
    conn = sqlite_oracle.make_db(path, ids, rows)
    gone = np.concatenate([np.arange(11, 40), rng.choice(np.arange(100, n + 1), 600, replace=False)])
    qs = [rows[10], rows[gone[0] - 1], rows[2500], rng.integers(0, 256, d, dtype=np.uint8)]
    eng = Engine.open(path)
    try:
        eng.remove_images(gone)
        assert len(eng.corpus) == n - len(gone)
        for round_ in range(2):
            for md in (1e3, 0.05):
                eng.max_distance_from_query = md
                for q in qs:
                    eng.query_by_image_hash_from_image(IndexedImage(visual_hash=bytes(q)))
                    got = eng.get_query_results()
                    want = sqlite_oracle.query(conn, bytes(q), md, 100)
                    assert [g.id for g in got] == [w[0] for w in want], (round_, md)
                    assert [g.distance_from_query for g in got] == [w[1] for w in want]
                    assert not set(gone.tolist()).intersection(g.id for g in got)
            eng.close()
            eng = Engine.open(path)                   # the file is the durable state: the same answers after re-opening
            assert len(eng.corpus) == n - len(gone)
    finally:
        eng.close()
        conn.close()
