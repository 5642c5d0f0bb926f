"""pbx_corpus_replace / pbx_sharded_replace: after a replacement every search path returns exactly what a corpus freshly
loaded with the updated table, in the same row order, returns (count, ids and their order, dist bit for bit, dot, norm2);
rows keep their positions; and the replacement is atomic with respect to searches, including device searches already
enqueued on other streams."""
import ctypes
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus, _replace
from tests import page_oracle
from tests.test_gpu_concurrency import DevOut, Oracle, hold, run_threads, to_dev

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def test_replace_argument_errors_need_no_gpu():
    L = nat.lib()
    ids = np.array([1, 2], np.int64)
    rows = np.zeros((2, 8), np.uint8)
    out = ctypes.c_uint64(7)
    assert L.pbx_corpus_replace(None, nat.ptr(ids), nat.ptr(rows), 2, ctypes.byref(out)) == -1 and out.value == 0
    assert L.pbx_corpus_replace(None, None, None, 2, None) == -1
    assert L.pbx_corpus_replace(None, None, None, 0, None) == -1                  # a NULL corpus is invalid even for n = 0
    out.value = 7
    assert L.pbx_sharded_replace(None, nat.ptr(ids), nat.ptr(rows), 2, ctypes.byref(out)) == -1 and out.value == 0
    assert L.pbx_sharded_replace(None, None, nat.ptr(rows), 1, None) == -1
    # shapes are checked before the library is called: the handle is never used
    fn = L.pbx_corpus_replace
    with pytest.raises(nat.PbxError) as e:
        _replace(fn, None, 8, ids, np.zeros((2, 7), np.uint8))                    # a row that is not dim bytes wide
    assert e.value.code == -2
    with pytest.raises(nat.PbxError) as e:
        _replace(fn, None, 8, ids, np.zeros((3, 8), np.uint8))                    # 2 ids, 3 rows
    assert e.value.code == -1
    with pytest.raises(nat.PbxError) as e:
        _replace(fn, None, 8, ids[:1], np.zeros(9, np.uint8))
    assert e.value.code == -2


# ---- helpers ------------------------------------------------------------------------------------------------------------
def same(res, want):
    o_ids, o_dist, o_dot, o_n2 = want
    return (len(res.ids) == len(o_ids) and list(res.ids) == list(o_ids)
            and np.array_equal(res.dist.view(np.uint32), np.asarray(o_dist, np.float32).view(np.uint32))
            and np.array_equal(res.dot, o_dot) and np.array_equal(res.norm2, o_n2))


def same_res(a, b):
    return same(a, (b.ids, b.dist, b.dot, b.norm2))


def clustered(rng, n, d, spread=3, centres=30):
    cent = rng.integers(0, 256, size=(centres, d))
    return np.clip(cent[rng.integers(0, centres, n)] + rng.integers(-spread, spread + 1, size=(n, d)), 0, 255).astype(np.uint8)


def corpus_rows(kind, rng, n, d):
    return clustered(rng, n, d) if kind == "clustered" else rng.integers(0, 256, size=(n, d), dtype=np.uint8)


def updated(ids, rows, req_ids, req_rows):
    """The table after `UPDATE ... SET hash = ? WHERE image_id = ?` per (id, row), in order."""
    last = {i: j for j, i in enumerate(np.asarray(req_ids).tolist())}          # a later statement overwrites an earlier one
    at = np.array([last.get(i, -1) for i in ids.tolist()], np.int64)
    new = rows.copy()
    new[at >= 0] = req_rows[at[at >= 0]]
    return new


def check_rows(c, ids, want_rows):
    got_ids, got_rows = c.read_rows(0, len(ids))
    assert np.array_equal(got_ids, ids) and np.array_equal(got_rows, want_rows)
    assert len(c) == len(ids)


# ---- parity on the single-query path, with filters, pages and the forced exact pass ----------------------------------------
@gpu
@pytest.mark.parametrize("kind", ["random", "clustered"])
@pytest.mark.parametrize("d", [8, 100, 256, 1000])
def test_parity_after_replace(d, kind):
    rng = np.random.default_rng(1000 + d + (kind == "clustered"))
    n = 6000
    rows = corpus_rows(kind, rng, n, d)
    ids = (rng.permutation(np.arange(1, n + 1)) * 3).astype(np.int64)
    for m in (1, 37, n // 10, n):
        pick = rng.choice(n, m, replace=False)
        req_ids = ids[pick]
        req_rows = corpus_rows(kind, rng, m, d)
        new = updated(ids, rows, req_ids, req_rows)
        allowed = rng.random(n) < 0.5
        with Corpus(d, capacity_hint=n) as c:
            c.load(ids, rows)
            assert c.replace(req_ids, req_rows) == m
            check_rows(c, ids, new)
            # the new hashes (the replaced rows must come first), the old ones (their bytes must be gone), a random one
            queries = np.concatenate([req_rows[[0, -1]], rows[pick[[0, -1]]], rng.integers(0, 256, size=(1, d), dtype=np.uint8)])
            for slack in (0, 1):
                c.set_candidate_slack(slack)
                for k, md in ((10, 1e3), (100, 1e3), (100, 0.05)):
                    for j, q in enumerate(queries):
                        got = c.search(q, k, md)[0]
                        assert same(got, oracle.topk(new, ids, q, k, md, threads=4)), f"m={m} slack={slack} k={k} md={md} q={j}"
                        if j < 2 and md > 1:
                            assert req_ids[[0, -1][j]] in got.ids.tolist()
            c.set_candidate_slack(0)
            for j, q in enumerate(queries[[0, 2, 4]]):
                for key, mask in (("within", allowed), ("excluding", ~allowed)):
                    sel = ids[allowed]
                    got = c.search(q, 50, 1e3, **{key: sel})[0]
                    assert same(got, page_oracle.page(new, ids, q, 50, 1e3, allowed=mask)), f"m={m} {key} q={j}"
                cursor = None
                for p in range(3):                          # three pages of 40
                    got = c.search(q, 40, 1e3, after=None if cursor is None else [cursor])[0]
                    assert same(got, page_oracle.page(new, ids, q, 40, 1e3, cursor=cursor)), f"m={m} page {p} q={j}"
                    if len(got.ids):
                        cursor = (float(got.dist[-1]), int(got.ids[-1]))


# ---- the tensor-core batched path ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", [64, 256])
def test_batched_path_after_replacing_10_percent(d):
    rng = np.random.default_rng(900 + d)
    n = 200_000
    rows = clustered(rng, n, d, spread=4, centres=200)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    pick = rng.choice(n, n // 10, replace=False)
    req_rows = clustered(rng, len(pick), d, spread=4, centres=50)
    new = updated(ids, rows, ids[pick], req_rows)
    with Corpus(d) as c, Corpus(d) as fresh:
        c.load(ids, rows)
        assert c.replace(ids[pick], req_rows) == len(pick)
        fresh.load(ids, new)
        queries = np.concatenate([req_rows[:64], rows[pick[:32]], rng.integers(0, 256, size=(64, d), dtype=np.uint8)])
        for k, md in ((100, 1e3), (10, 0.05)):
            before = c.stats().batched_queries
            got = c.search(queries, k, md)
            assert c.stats().batched_queries == before + len(queries)
            ref = fresh.search(queries, k, md)
            for i in range(len(queries)):
                assert same_res(got[i], ref[i]), (k, md, i)
            for i in list(range(0, len(queries), 23)) + [0, 64]:
                assert same(got[i], oracle.topk(new, ids, queries[i], k, md, threads=8)), (k, md, i)
        c.set_candidate_slack(1)                          # every query takes the exact pass
        fresh.set_candidate_slack(1)
        got, ref = c.search(queries[:32], 100, 1e3), fresh.search(queries[:32], 100, 1e3)
        for i in range(32):
            assert same_res(got[i], ref[i]), i


# ---- the 32-row block bounds of the batched epilogue ----------------------------------------------------------------------
def tiny_rows(rng, m, d):
    """Bytes 127 / 128: norm^2 = d, the smallest a row can have, and row term 0."""
    return np.where(rng.random((m, d)) < 0.5, 127, 128).astype(np.uint8)


@gpu
def test_written_row_outside_its_block_bounds_is_found_by_the_batched_path():
    """Without the block metadata step, a written row keeps its block's old {norm, rowterm} range, which the batched
    epilogue trusts as a bound.  (1) A block of tiny-norm rows receives a high-norm row (the query itself): the stale range
    says no row of the block can reach it.  (2) A row of a block of maximal-norm rows (bytes 255 / 0) becomes a tiny-norm
    row."""
    rng = np.random.default_rng(23)
    n, d = 60_000, 64
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    rows[320:352] = tiny_rows(rng, 32, d)                                  # block 10: tiny norms
    rows[640:672] = np.where(rng.random((32, d)) < 0.5, 0, 255)             # block 20: the largest norms
    ids = np.arange(1, n + 1, dtype=np.int64)
    q_high = rng.integers(0, 256, size=(1, d), dtype=np.uint8)
    q_tiny = tiny_rows(rng, 1, d)
    req_ids, req_rows = np.array([331, 651], np.int64), np.concatenate([q_high, q_tiny])     # rows 330 and 650
    new = updated(ids, rows, req_ids, req_rows)
    queries = np.concatenate([q_high, q_tiny, rng.integers(0, 256, size=(30, d), dtype=np.uint8)])
    with Corpus(d) as c:
        c.load(ids, rows)
        assert c.replace(req_ids, req_rows) == 2
        check_rows(c, ids, new)
        before = c.stats().batched_queries
        got = c.search(queries, 10, 1e3)
        assert c.stats().batched_queries == before + len(queries)
        assert got[0].ids[0] == 331 and got[0].dist[0] <= 1e-6
        assert got[1].ids[0] == 651 and got[1].dist[0] <= 1e-6
        for i in range(len(queries)):
            assert same(got[i], oracle.topk(new, ids, queries[i], 10, 1e3, threads=8)), i


# ---- semantics ------------------------------------------------------------------------------------------------------------
@gpu
def test_replace_semantics():
    rng = np.random.default_rng(3)
    d = 32
    n = 3000
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = np.arange(1, n + 1, dtype=np.int64)
    ids[[10, 500, 2999]] = 77                                              # one id on four rows (76 is the fourth)
    L = nat.lib()
    with Corpus(d, capacity_hint=8192) as c:
        out = ctypes.c_uint64(9)
        assert c.replace([1, 2], rows[:2]) == 0 and len(c) == 0                # empty corpus
        c.load(ids, rows)
        cap = c.stats().capacity_rows
        assert L.pbx_corpus_replace(c.handle, None, nat.ptr(rows), 1, None) == -1
        assert L.pbx_corpus_replace(c.handle, nat.ptr(ids), None, 1, ctypes.byref(out)) == -1 and out.value == 0
        out.value = 9
        assert L.pbx_corpus_replace(c.handle, None, None, 0, ctypes.byref(out)) == 0 and out.value == 0
        assert c.replace(np.zeros(0, np.int64), np.zeros((0, d), np.uint8)) == 0
        with pytest.raises(nat.PbxError) as e:
            c.replace([1], np.zeros((1, d + 1), np.uint8))
        assert e.value.code == -2
        with pytest.raises(nat.PbxError):
            c.replace([1, 2], rows[:1])
        # ids that match nothing are ignored and not counted
        assert c.replace([-5, 10**12, 0], rows[:3]) == 0
        check_rows(c, ids, rows)
        # an id on several rows: all of them; an id repeated in the request: its last hash; a row whose new hash equals
        # its old one still counts
        new_rows = rng.integers(0, 256, size=(5, d), dtype=np.uint8)
        req_ids = np.array([77, 5, 40, 5, 40], np.int64)
        req = np.concatenate([new_rows[:4], rows[ids == 40]])
        assert c.replace(req_ids, req) == 4 + 1 + 1
        want = updated(ids, rows, req_ids, req)
        assert np.array_equal(want[[10, 76, 500, 2999]], np.repeat(new_rows[:1], 4, axis=0))
        assert np.array_equal(want[ids == 5][0], new_rows[3]) and np.array_equal(want[ids == 40][0], rows[ids == 40][0])
        check_rows(c, ids, want)
        assert c.stats().capacity_rows == cap
        for q in (new_rows[0], new_rows[1], new_rows[3], rows[4]):
            got = c.search(q, 10, 1e7)[0]
            assert same(got, oracle.topk(want, ids, q, 10, 1e7)), q[:4]
        assert list(c.search(new_rows[0], 3, 1e3)[0].ids) == [77, 77, 77]


# ---- interplay with appends and removal -----------------------------------------------------------------------------------
@gpu
def test_replace_pending_moved_and_sequenced_rows():
    rng = np.random.default_rng(5)
    n, d = 20_000, 64
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = np.arange(1, n + 1, dtype=np.int64)
    with Corpus(d, capacity_hint=32768) as c:
        c.load(ids, rows)
        # pending (coalesced, not flushed) appends are subject to the replacement
        extra = rng.integers(0, 256, size=(10, d), dtype=np.uint8)
        c.append(np.arange(50_001, 50_011), extra)                            # fewer than 64 rows: coalesced, pending
        assert len(c) == n + 10
        t_ids, t_rows = np.concatenate([ids, np.arange(50_001, 50_011)]), np.concatenate([rows, extra])
        r1 = rng.integers(0, 256, size=(3, d), dtype=np.uint8)
        assert c.replace([50_003, 50_010, 7], r1) == 3
        t_rows = updated(t_ids, t_rows, np.array([50_003, 50_010, 7]), r1)
        check_rows(c, t_ids, t_rows)
        # a row that a removal moved into a hole is found by id
        gone = np.isin(t_ids, [2, 3])
        assert c.remove([2, 3]) == 2
        nk = len(t_ids) - 2
        holes = np.flatnonzero(gone[:nk])
        srcs = nk + np.flatnonzero(~gone[nk:])
        t_ids, t_rows = t_ids.copy(), t_rows.copy()
        t_ids[holes], t_rows[holes] = t_ids[srcs], t_rows[srcs]
        t_ids, t_rows = t_ids[:nk], t_rows[:nk]
        assert set(t_ids[holes].tolist()) == {50_010, 50_009}
        r2 = rng.integers(0, 256, size=(1, d), dtype=np.uint8)
        assert c.replace([50_010], r2) == 1
        t_rows = updated(t_ids, t_rows, np.array([50_010]), r2)
        check_rows(c, t_ids, t_rows)
        # replace, then remove, then append, in sequence
        r3 = rng.integers(0, 256, size=(2, d), dtype=np.uint8)
        assert c.replace([100, 200], r3) == 2
        t_rows = updated(t_ids, t_rows, np.array([100, 200]), r3)
        assert c.remove([100]) == 1
        keep = t_ids != 100
        nk = len(t_ids) - 1
        hole = int(np.flatnonzero(~keep)[0])
        if hole < nk:
            t_ids[hole], t_rows[hole] = t_ids[nk], t_rows[nk]
        t_ids, t_rows = t_ids[:nk], t_rows[:nk]
        r4 = rng.integers(0, 256, size=(1, d), dtype=np.uint8)
        c.append([100], r4)
        t_ids, t_rows = np.concatenate([t_ids, [100]]), np.concatenate([t_rows, r4])
        check_rows(c, t_ids, t_rows)
        queries = np.concatenate([r1, r2, r3, r4, rows[[99, 199]], rng.integers(0, 256, size=(24, d), dtype=np.uint8)])
        for i, q in enumerate(queries[:8]):
            assert same(c.search(q, 20, 1e3)[0], oracle.topk(t_rows, t_ids, q, 20, 1e3, threads=4)), i
        got = c.search(queries, 20, 1e3)
        for i, q in enumerate(queries):
            assert same(got[i], oracle.topk(t_rows, t_ids, q, 20, 1e3, threads=4)), i


# ---- atomicity ------------------------------------------------------------------------------------------------------------
@gpu
def test_replace_orders_after_device_searches_on_held_streams():
    import torch
    n, d, k, md = 120_000, 64, 50, 1e3
    rng = np.random.default_rng(61)
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    pick = rng.choice(n, 20_000, replace=False)
    req_rows = rng.integers(0, 256, size=(len(pick), d), dtype=np.uint8)
    new = updated(ids, rows, ids[pick], req_rows)
    queries = np.concatenate([rows[pick[:8]], req_rows[:8]])              # old bytes vanish, new bytes appear
    pre, post = Oracle(rows, ids), Oracle(new, ids)
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    dq = to_dev(queries)
    shape = (("A", 1), ("B", 16), ("corpus", 16), ("A", 16), ("B", 1), ("corpus", 1))
    out_sets = [[DevOut(nq, k) for _, nq in shape] for _ in range(3)]

    def calls(orc, outs):
        out = []
        for (where, nq), o in zip(shape, outs):
            stream = None if where == "corpus" else (A if where == "A" else B).cuda_stream
            c.search_device(dq.data_ptr(), nq, k, md, *o.ptrs(), stream)
            out.append((where, nq, o, orc))
        return out

    def check(enqueued, when):
        for where, nq, o, orc in enqueued:
            for i, g in enumerate(o.results()):
                assert same(g, orc(queries[i], k, md)), f"{when} the replacement: {where} nq={nq} query {i}"

    with Corpus(d) as c:
        c.load(ids, rows)
        torch.cuda.synchronize()
        calls(pre, out_sets[0])                           # warm-up: scratch at its size
        c.synchronize()
        torch.cuda.synchronize()
        hold(A)
        hold(B)
        before = calls(pre, out_sets[1])
        assert not A.query() and not B.query()
        assert c.replace(ids[pick], req_rows) == len(pick)                   # no synchronisation before this
        assert A.query() and B.query(), "the replacement returned before the searches enqueued ahead of it had finished"
        after = calls(post, out_sets[2])
        c.synchronize()
        torch.cuda.synchronize()
        check(before, "before")
        check(after, "after")


@gpu
def test_host_searches_see_all_of_a_replacement_or_none():
    """One thread runs a series of replacements while another makes host searches (single and batched): every answer is
    the oracle's answer over one of the table states the series passes through."""
    n, d, k = 200_000, 64, 20
    rng = np.random.default_rng(71)
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    steps = [rng.choice(n, m, replace=False) for m in (1, 5000, 40, 20_000)]
    tables = [rows]
    reqs = []
    for pick in steps:
        r = rng.integers(0, 256, size=(len(pick), d), dtype=np.uint8)
        reqs.append((ids[pick], r))
        tables.append(updated(ids, tables[-1], ids[pick], r))
    queries = np.concatenate([tables[0][steps[0]], tables[1][steps[0]], tables[3][steps[2][:2]], tables[4][steps[3][:2]],
                              rng.integers(0, 256, size=(2, d), dtype=np.uint8)])
    states = [Oracle(t, ids) for t in tables]
    for st in states:
        for q in queries:
            st(q, k)
    seen = []
    started, done = threading.Event(), threading.Event()

    def writer():
        try:
            started.wait(60)
            for r_ids, r_rows in reqs:
                assert c.replace(r_ids, r_rows) == len(r_ids)
        finally:
            done.set()

    def reader():
        r = 0
        while not done.is_set() or r < 24:
            if r % 2 == 0:
                qi = (r // 2) % len(queries)
                seen.append(([qi], c.search(queries[qi], k)))
            else:
                seen.append((list(range(len(queries))), c.search(queries, k)))
            r += 1
            if r == 4:
                started.set()
        started.set()

    with Corpus(d) as c:
        c.load(ids, rows)
        c.search(queries[0], k)
        c.search(queries, k)
        run_threads([writer, reader])
        hit = set()
        for j, (qis, res) in enumerate(seen):
            match = [st for st in range(len(states)) if all(same(res[i], states[st](queries[qi], k)) for i, qi in enumerate(qis))]
            assert match, f"search {j} matches no table state"
            hit.update(match)
        assert 0 in hit, hit                              # searches ran before the first replacement
        for qi, q in enumerate(queries):
            assert same(c.search(q, k)[0], states[-1](q, k)), qi


# ---- several shards --------------------------------------------------------------------------------------------------------
def devices(n):
    have = max(1, nat.lib().pbx_device_count())
    return [i % have for i in range(n)]


@gpu
def test_multi_device_corpus_replace():
    rng = np.random.default_rng(41)
    n, d = 60_000, 256
    rows = clustered(rng, n, d, spread=2, centres=40)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 3
    ids[n - 1] = ids[5]                                   # one id in shard 0 and in shard 2
    pick = np.concatenate([[5, 21_000, 45_000], rng.choice(np.setdiff1d(np.arange(n - 1), [5, 21_000, 45_000]), 3000, replace=False)])
    req_ids = ids[pick]
    req_rows = clustered(rng, len(req_ids), d, spread=2, centres=10)
    new = updated(ids, rows, req_ids, req_rows)
    expect = int(np.isin(ids, req_ids).sum())
    queries = np.concatenate([req_rows[:3], rows[pick[:3]], rng.integers(0, 256, size=(20, d), dtype=np.uint8)])
    with MultiDeviceCorpus(d, devices(3)) as mc:
        mc.load(ids, rows)
        assert mc.replace(req_ids, req_rows) == expect and len(mc) == n
        for k, md, qs in ((100, 1e3, queries), (300, 1e7, queries[:2]), (10, 0.02, queries[:6])):
            got = mc.search(qs, k, md)
            for qi, q in enumerate(qs):
                assert same(got[qi], oracle.topk(new, ids, q, k, md, threads=8)), (k, md, qi)
        assert list(mc.search(req_rows[0], 2, 1e3)[0].ids) == [ids[5], ids[5]]


@gpu
def test_sharded_corpus_replace_between_processes_sharing_one_gpu():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29673", os.path.join(ROOT, "tools", "replace_exchange_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "replace_exchange_check OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


# ---- the Engine mirror ---------------------------------------------------------------------------------------------------
@gpu
def test_engine_update_image_hashes_matches_verbatim_sql(tmp_path):
    from pixelbox_b200.engine import Engine, IndexedImage
    from tests import sqlite_oracle
    rng = np.random.default_rng(8)
    n, d = 4000, 64
    rows = clustered(rng, n, d)
    ids = np.arange(1, n + 1, dtype=np.int64)
    path = str(tmp_path / "replace.db")
    conn = sqlite_oracle.make_db(path, ids, rows)
    pick = rng.choice(np.arange(1, n + 1), 300, replace=False)
    new = clustered(rng, len(pick), d)
    pairs = [(int(i), bytes(h)) for i, h in zip(pick, new)]
    pairs.append((int(pick[0]), bytes(rows[7])))                        # the last UPDATE of an id wins
    pairs.append((10**9, bytes(new[1])))                                 # no semantic_hashes row: nothing changes
    pairs.append((int(pick[1]), bytes(d + 3)))                           # a length the corpus cannot hold: leaves the device
    bad = int(pick[1])
    qs = [new[0], rows[7], new[1], rows[pick[2] - 1], new[5], rng.integers(0, 256, d, dtype=np.uint8)]

    def sql(q, md):
        """The verbatim SQL, without the row whose hash the corpus cannot represent (the UDF would zip-truncate it)."""
        return [w for w in sqlite_oracle.query(conn, bytes(q), md, 101) if w[0] != bad][:100]

    eng = Engine.open(path)
    try:
        assert eng.skipped_rows == 0
        eng.update_image_hashes(pairs)
        assert eng.skipped_rows == 1 and len(eng.corpus) == n - 1
        assert conn.execute("SELECT COUNT(*) FROM semantic_hashes").fetchone()[0] == n
        for round_ in range(2):
            for md in (1e3, 0.05):
                eng.max_distance_from_query = md
                for q in qs:
                    eng.query_by_image_hash_from_image(IndexedImage(visual_hash=bytes(q)))
                    got = eng.get_query_results()
                    want = sql(q, md)
                    assert [g.id for g in got] == [w[0] for w in want], (round_, md)
                    assert [g.distance_from_query for g in got] == [w[1] for w in want]
            eng.close()
            eng = Engine.open(path)                   # the file is the durable state: the same answers after re-opening
            assert eng.skipped_rows == 1 and len(eng.corpus) == n - 1
        # the skipped row gets a hash of the corpus' dim again: it returns to the device
        eng.update_image_hashes([(int(pick[1]), bytes(new[1]))])
        assert eng.skipped_rows == 0 and len(eng.corpus) == n
        eng.query_by_image_hash_from_image(IndexedImage(visual_hash=bytes(new[1])))
        want = sqlite_oracle.query(conn, bytes(new[1]), eng.max_distance_from_query, 100)       # every hash has dim bytes again
        assert [g.id for g in eng.get_query_results()] == [w[0] for w in want] and want[0][0] == int(pick[1])
    finally:
        eng.close()
        conn.close()
