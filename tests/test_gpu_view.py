"""Views (pbx_corpus_view_create / pbx_sharded_view_create): a search on a view returns exactly what the filtered search
(PBX_FILTER_INCLUDE, the view's set) returns on the parent at that moment, on every path, and the view follows every
change of its parent.  Each answer is compared field by field (count, ids and their order, dist bits, dot, norm2) with
the filtered search on the parent, with a corpus freshly loaded with only the allowed rows, and with the CPU oracle where
the size allows.  Rows with equal (dist, image_id) -- an id on several rows -- are compared as multisets."""
import ctypes
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus, SearchResult
from tests import page_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


# ---- argument errors (no GPU needed) --------------------------------------------------------------------------------------
def test_view_argument_errors_need_no_gpu():
    L = nat.lib()
    ids = np.array([1, 2], np.int64)
    h = ctypes.c_void_p(5)
    out = ctypes.c_uint64(7)
    assert L.pbx_corpus_view_create(None, nat.ptr(ids), 2, ctypes.byref(h)) == -1 and not h.value
    assert L.pbx_corpus_view_create(None, nat.ptr(ids), 2, None) == -1
    assert L.pbx_corpus_view_add(None, nat.ptr(ids), 2, ctypes.byref(out)) == -1 and out.value == 0
    out.value = 7
    assert L.pbx_corpus_view_drop(None, nat.ptr(ids), 2, ctypes.byref(out)) == -1 and out.value == 0
    h.value = 5
    assert L.pbx_sharded_view_create(None, nat.ptr(ids), 2, ctypes.byref(h)) == -1 and not h.value
    assert L.pbx_sharded_view_create(None, nat.ptr(ids), 2, None) == -1
    assert L.pbx_sharded_view_add(None, nat.ptr(ids), 2, None) == -1
    assert L.pbx_sharded_view_drop(None, nat.ptr(ids), 2, None) == -1
    assert b"NULL" in L.pbx_last_error()


# ---- helpers ------------------------------------------------------------------------------------------------------------
def fields(r):
    return r.ids, r.dist, r.dot, r.norm2


def same(res, want):
    """Field by field; rows with equal (dist, image_id) may come in any order (an id on several rows)."""
    o_ids, o_dist, o_dot, o_n2 = (np.asarray(x) for x in want)
    if len(res.ids) != len(o_ids) or list(res.ids) != list(o_ids):
        return False
    if not np.array_equal(res.dist.view(np.uint32), np.asarray(o_dist, np.float32).view(np.uint32)):
        return False
    a = sorted(zip(res.dist.view(np.uint32).tolist(), res.ids.tolist(), res.dot.tolist(), res.norm2.tolist()))
    b = sorted(zip(np.asarray(o_dist, np.float32).view(np.uint32).tolist(), o_ids.tolist(), o_dot.tolist(), o_n2.tolist()))
    return a == b


def clustered(rng, n, d, spread=3, centres=30):
    cent = rng.integers(0, 256, size=(centres, d))
    return np.clip(cent[rng.integers(0, centres, n)] + rng.integers(-spread, spread + 1, size=(n, d)), 0, 255).astype(np.uint8)


def id_set(kind, rng, ids):
    n = len(ids)
    if kind == "empty":
        return np.zeros(0, np.int64)
    if kind == "one":
        return ids[[n // 2]]
    if kind == "1000":
        return rng.choice(ids, 1000, replace=False)
    if kind == "1pct":
        return ids[rng.random(n) < 0.01]
    if kind == "50pct":
        return ids[rng.random(n) < 0.5]
    # ids absent from the corpus, and ids repeated in the request
    pick = rng.choice(ids, 300, replace=False)
    return np.concatenate([pick, pick[:100], [-5, 0, 10 ** 12], pick[::7]]).astype(np.int64)


def check_view(view, parent, fset, table_rows, table_ids, queries, ks=((100, 1e3), (10, 1e3), (100, 0.05)), oracle_check=True,
               fresh_check=True):
    """Every query of `queries`, single and as one batch: view == filtered parent == fresh corpus == oracle."""
    allowed = np.isin(table_ids, fset)
    a_rows, a_ids = table_rows[allowed], table_ids[allowed]
    fresh = None
    if fresh_check:
        fresh = Corpus(view.dim, capacity_hint=max(len(a_ids), 1))
        fresh.load(a_ids, a_rows)
    try:
        for k, md in ks:
            batch_v = view.search(queries, k, md)
            batch_p = parent.search(queries, k, md, within=fset)
            batch_f = fresh.search(queries, k, md) if fresh else None
            for j, q in enumerate(queries):
                single = view.search(q, k, md)[0]
                want = fields(parent.search(q, k, md, within=fset)[0])
                assert same(single, want), f"single k={k} md={md} q={j}"
                assert same(batch_v[j], fields(batch_p[j])), f"batch k={k} md={md} q={j}"
                assert same(batch_v[j], want), f"batch vs single k={k} md={md} q={j}"
                if fresh:
                    assert same(single, fields(batch_f[j])), f"fresh k={k} md={md} q={j}"
                if oracle_check and j < 3:
                    assert same(single, oracle.topk(a_rows, a_ids, q, k, md, threads=oracle.max_threads())), f"oracle k={k} md={md} q={j}"
    finally:
        if fresh:
            fresh.close()


def table(seed, n, d, kind="clustered"):
    rng = np.random.default_rng(seed)
    rows = clustered(rng, n, d) if kind == "clustered" else rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = (rng.permutation(np.arange(1, n + 1)) * 3).astype(np.int64)
    return rng, rows, ids


# ---- parity of a fresh view ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind", ["empty", "one", "1000", "1pct", "50pct", "absent+repeated"])
@pytest.mark.parametrize("d", [8, 64, 100, 256])
def test_view_parity(d, kind):
    rng, rows, ids = table(7000 + d, 20_000, d)
    fset = id_set(kind, rng, ids)
    queries = np.concatenate([rows[rng.choice(len(rows), 6)], rng.integers(0, 256, size=(2, d), dtype=np.uint8)])
    if len(fset):
        allowed_rows = rows[np.isin(ids, fset)]
        queries = np.concatenate([queries, allowed_rows[:2]])
    with Corpus(d, capacity_hint=len(ids)) as c:
        c.load(ids, rows)
        with c.view(fset) as v:
            assert len(v) == int(np.isin(ids, fset).sum())
            got_ids, got_rows = v.read_rows(0, len(v))
            sel = np.isin(ids, fset)
            assert np.array_equal(got_ids, ids[sel]) and np.array_equal(got_rows, rows[sel])     # parent row order at build
            b0 = v.stats().batched_queries
            check_view(v, c, fset, rows, ids, queries)
            if kind == "50pct" and d in (64, 256):
                assert v.stats().batched_queries > b0, "the batched path did not run on the view"
            # the forced exact pass on both sides
            v.set_candidate_slack(1)
            c.set_candidate_slack(1)
            x0 = v.stats().exact_passes
            check_view(v, c, fset, rows, ids, queries[:4], ks=((100, 1e3),), oracle_check=False, fresh_check=False)
            if kind == "50pct":
                assert v.stats().exact_passes > x0


@gpu
def test_view_one_id_on_several_rows_and_plateau():
    rng, rows, ids = table(71, 12_000, 64)
    ids[100:140] = ids[100]                     # one id on 40 rows (differing rows)
    rows[2000:2600] = rows[2000]                # a plateau of 600 identical rows, half of them in the set
    ids[5000:5020] = ids[5000]
    rows[5000:5020] = rows[5000]                # one id on 20 identical rows
    fset = np.concatenate([ids[[100, 5000]], ids[2000:2300], ids[rng.random(len(ids)) < 0.2]])
    queries = np.stack([rows[100], rows[120], rows[2000], rows[5000], rows[7]])
    with Corpus(64, capacity_hint=len(ids)) as c:
        c.load(ids, rows)
        with c.view(fset) as v:
            check_view(v, c, fset, rows, ids, queries, ks=((100, 1e3), (10, 1e3), (500, 1e3), (2048, 1e7)))
            # a removal moves the view's rows: order within equal (dist, id) may change, nothing else
            gone = ids[rng.random(len(ids)) < 0.1]
            c.remove(gone)
            keep = ~np.isin(ids, gone)
            check_view(v, c, fset, rows[keep], ids[keep], queries, ks=((100, 1e3), (500, 1e3)))


# ---- pages, device forms, a filter on a view ------------------------------------------------------------------------------
def chain_pages(search, q, k, md, depth):
    """Pages of k after the last row of the previous page until `depth` rows or the end: one concatenated list."""
    out, cur = [], None
    while sum(len(r.ids) for r in out) < depth:
        r = search(q, k, md, after=[cur])[0]
        out.append(r)
        if len(r.ids) < k:
            break
        cur = (float(r.dist[-1]), int(r.ids[-1]))
    cat = lambda f: np.concatenate([getattr(r, f) for r in out])            # noqa: E731
    return cat("ids"), cat("dist"), cat("dot"), cat("norm2")


@gpu
@pytest.mark.parametrize("d", [64, 100])
def test_view_pages_past_max_k(d):
    rng, rows, ids = table(72 + d, 30_000, d)
    fset = ids[rng.random(len(ids)) < 0.5]
    allowed = np.isin(ids, fset)
    with Corpus(d, capacity_hint=len(ids)) as c:
        c.load(ids, rows)
        with c.view(fset) as v:
            with Corpus(d, capacity_hint=int(allowed.sum())) as fresh:
                fresh.load(ids[allowed], rows[allowed])
                for qi, q in enumerate((rows[3], rng.integers(0, 256, d, dtype=np.uint8))):
                    for k in (1000, 2048):
                        got = chain_pages(lambda *a, **kw: v.search(*a, **kw), q, k, 1e3, 5000)
                        want = chain_pages(lambda *a, **kw: c.search(*a, within=fset, **kw), q, k, 1e3, 5000)
                        frs = chain_pages(lambda *a, **kw: fresh.search(*a, **kw), q, k, 1e3, 5000)
                        o = page_oracle.page(rows, ids, q, 5000, 1e3, allowed=allowed)
                        msg = f"q={qi} k={k} rows: view {len(got[0])} filtered {len(want[0])} fresh {len(frs[0])} oracle {len(o[0])}"
                        assert same(SearchResult(*got), want), msg
                        assert same(SearchResult(*got), frs), msg
                        # past PBX_MAX_K; the oracle decides the length (rows with dist >= max_dist end the chain early)
                        assert len(got[0]) > nat.PBX_MAX_K, msg
                        assert same(SearchResult(*(x[:5000] for x in got)), o), msg
            # a filter on the view intersects with the view's set
            sub = np.concatenate([fset[::3], ids[~allowed][:500]])
            for q in (rows[3], rows[4]):
                assert same(v.search(q, 100, 1e3, within=sub)[0], fields(c.search(q, 100, 1e3, within=np.intersect1d(sub, fset))[0]))
                assert same(v.search(q, 100, 1e3, excluding=sub)[0], fields(c.search(q, 100, 1e3, within=np.setdiff1d(fset, sub))[0]))


@gpu
def test_view_device_form_pipeline():
    import torch
    from tests.test_gpu_concurrency import DevOut, to_dev
    rng, rows, ids = table(73, 20_000, 256)
    fset = ids[rng.random(len(ids)) < 0.3]
    queries = np.concatenate([rows[rng.choice(len(rows), 5)], rng.integers(0, 256, size=(3, 256), dtype=np.uint8)])
    nq, k = len(queries), 100
    with Corpus(256, capacity_hint=len(ids)) as c:
        c.load(ids, rows)
        with c.view(fset) as v:
            d_q = to_dev(queries)
            s = torch.cuda.Stream()
            outs = [DevOut(nq, k) for _ in range(3)]
            with torch.cuda.stream(s):
                v.search_device(d_q.data_ptr(), nq, k, 1e3, *outs[0].ptrs(), stream=s.cuda_stream)
                # the next pages: each query's cursor is the last record of its previous page (all pages are full)
                for p in (1, 2):
                    cur = outs[p - 1].hits.view(nq, k * nat.HIT_DTYPE.itemsize)[:, (k - 1) * 24:k * 24].contiguous()
                    v.search_device_page(d_q.data_ptr(), nq, k, 1e3, *outs[p].ptrs(), d_after_ptr=cur.data_ptr(), stream=s.cuda_stream)
            s.synchronize()
            pages = [o.results() for o in outs]
            for j, q in enumerate(queries):
                want = chain_pages(lambda *a, **kw: c.search(*a, within=fset, **kw), q, k, 1e3, 3 * k)
                got = [np.concatenate([fields(pages[p][j])[f] for p in range(3)]) for f in range(4)]
                assert [len(x) for x in got] == [3 * k] * 4
                for g, w in zip(got, want):
                    assert np.array_equal(g.view(np.uint32) if g.dtype == np.float32 else g, w.view(np.uint32) if w.dtype == np.float32 else w)


# ---- following the parent ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", [64, 100])
def test_view_follows_every_change(d):
    import torch
    rng, rows, ids = table(74 + d, 15_000, d)
    fset = np.concatenate([ids[rng.random(len(ids)) < 0.1], [10 ** 9 + 1, 10 ** 9 + 2, 10 ** 9 + 3]])   # three ids appended later
    queries = np.concatenate([rows[rng.choice(len(rows), 4)], rng.integers(0, 256, size=(2, d), dtype=np.uint8)])
    t_rows, t_ids = rows.copy(), ids.copy()
    with Corpus(d, capacity_hint=1000) as c:
        c.load(ids, rows)
        v = c.view(fset)
        cur = np.unique(fset)

        def state(msg):
            assert len(v) == int(np.isin(t_ids, cur).sum()), msg
            check_view(v, c, cur, t_rows, t_ids, queries, ks=((100, 1e3), (10, 0.05)), oracle_check=False)

        state("built")
        # appends in and out of the set: a bulk one, then single-row coalesced ones that are not flushed yet
        new_ids = np.array([10 ** 9 + 1, 10 ** 9 + 7] + list(range(2 * 10 ** 9, 2 * 10 ** 9 + 200)), np.int64)
        new_rows = np.concatenate([queries[:2], clustered(rng, 200, d)])
        c.append(new_ids, new_rows)
        t_rows, t_ids = np.concatenate([t_rows, new_rows]), np.concatenate([t_ids, new_ids])
        state("bulk append")
        one_ids = np.array([10 ** 9 + 2, 10 ** 9 + 8], np.int64)
        for i, r in zip(one_ids, queries[2:4]):
            c.append(np.array([i]), r.reshape(1, -1))
        t_rows, t_ids = np.concatenate([t_rows, queries[2:4]]), np.concatenate([t_ids, one_ids])
        # still pending in the parent: the view's search must upload them first
        got = v.search(queries[2], 10, 1e3)[0]
        assert 10 ** 9 + 2 in got.ids.tolist() and 10 ** 9 + 8 not in got.ids.tolist()
        state("coalesced append")
        # append_device
        dev_ids = np.array([10 ** 9 + 3, 10 ** 9 + 9], np.int64)
        dev_rows = clustered(rng, 2, d)
        d_i, d_r = torch.from_numpy(dev_ids).cuda(), torch.from_numpy(dev_rows).cuda()
        torch.cuda.synchronize()
        c.append_device(d_i.data_ptr(), d_r.data_ptr(), 2)
        t_rows, t_ids = np.concatenate([t_rows, dev_rows]), np.concatenate([t_ids, dev_ids])
        state("append_device")
        # a removal that moves view rows (ids early in the table, in and out of the set)
        gone = np.concatenate([cur[:30], t_ids[:200], [10 ** 9 + 1]])
        assert c.remove(gone) == int(np.isin(t_ids, gone).sum())
        keep = ~np.isin(t_ids, gone)
        t_rows, t_ids = t_rows[keep], t_ids[keep]
        state("remove")
        # a replacement of rows in and out of the view; the view's rows stay the parent's bytes
        pick = np.concatenate([cur[40:80], t_ids[~np.isin(t_ids, cur)][:40]])
        pick = pick[np.isin(pick, t_ids)]
        new = clustered(rng, len(pick), d)
        c.replace(pick, new)
        at = {int(i): j for j, i in enumerate(pick.tolist())}
        for r, i in enumerate(t_ids.tolist()):
            if i in at:
                t_rows[r] = new[at[i]]
        state("replace")
        vi, vr = v.read_rows(0, len(v))
        sel = np.isin(t_ids, cur)
        order = {int(i): r for r, i in zip(np.nonzero(sel)[0], t_ids[sel])}
        assert np.array_equal(vr, t_rows[[order[int(i)] for i in vi]])
        # view_add, view_drop, re-adding a dropped id
        add = t_ids[~np.isin(t_ids, cur)][:300]
        assert v.view_add(np.concatenate([add, add[:10], cur[:5]])) == len(add)
        cur = np.union1d(cur, add)
        state("view_add")
        drop = cur[::4]
        assert v.view_drop(drop) == int(np.isin(t_ids, drop).sum())
        cur = np.setdiff1d(cur, drop)
        state("view_drop")
        assert v.view_add(drop[:50]) == int(np.isin(t_ids, drop[:50]).sum())
        cur = np.union1d(cur, drop[:50])
        state("re-add")
        # load rebuilds the view from the new contents
        rng2, rows2, ids2 = table(75 + d, 9000, d)
        c.load(ids2, rows2)
        t_rows, t_ids = rows2, ids2
        state("load")
        with pytest.raises(nat.PbxError) as e:
            v.append(ids2[:1], rows2[:1])
        assert e.value.code == -1
        for call in (lambda: v.load(ids2[:1], rows2[:1]), lambda: v.remove(ids2[:1]), lambda: v.replace(ids2[:1], rows2[:1]),
                     lambda: v.fill_synthetic(10, 1), lambda: v.view(ids2[:1]), lambda: c.view_add(ids2[:1]), lambda: c.view_drop(ids2[:1])):
            with pytest.raises(nat.PbxError) as e:
                call()
            assert e.value.code == -1
        # the parent goes first: the view keeps its rows and stays searchable; view_add is refused, view_drop works
        want = [fields(c.search(q, 100, 1e3, within=cur)[0]) for q in queries]
        c.close()
        for q, w in zip(queries, want):
            assert same(v.search(q, 100, 1e3)[0], w)
        with pytest.raises(nat.PbxError) as e:
            v.view_add(ids2[:10])
        assert e.value.code == -1
        v.view_drop(cur[:10])
        v.close()


# ---- concurrency -------------------------------------------------------------------------------------------------------
@gpu
def test_view_searches_while_the_parent_changes():
    """Searches of the view from another thread (host form) and on another stream (device form) while the parent
    appends, removes and replaces: every answer is one of the table states, never a mix."""
    import torch
    from tests.test_gpu_concurrency import DevOut, to_dev
    rng, rows, ids = table(76, 20_000, 64)
    fset = ids[rng.random(len(ids)) < 0.2]
    queries = np.concatenate([rows[np.isin(ids, fset)][:3], rng.integers(0, 256, size=(1, 64), dtype=np.uint8)])
    k = 50
    # the table states: after each mutation of the plan
    plan, t_rows, t_ids = [], rows.copy(), ids.copy()
    states = [(t_rows, t_ids)]
    for step in range(6):
        if step % 3 == 0:
            a_ids = np.concatenate([fset[step * 5:step * 5 + 5] + 0, np.arange(5) + 10 ** 9 + 10 * step]).astype(np.int64)
            a_rows = np.concatenate([queries[:3], clustered(rng, 7, 64)])[:len(a_ids)]
            plan.append(("append", a_ids, a_rows))
            t_rows, t_ids = np.concatenate([t_rows, a_rows]), np.concatenate([t_ids, a_ids])
        elif step % 3 == 1:
            gone = np.concatenate([fset[100 + step * 20:120 + step * 20], t_ids[:50]])
            plan.append(("remove", gone, None))
            keep = ~np.isin(t_ids, gone)
            t_rows, t_ids = t_rows[keep], t_ids[keep]
        else:
            pick = fset[300 + step * 20:340 + step * 20]
            pick = pick[np.isin(pick, t_ids)]
            new = clustered(rng, len(pick), 64)
            plan.append(("replace", pick, new))
            at = {int(i): j for j, i in enumerate(pick.tolist())}
            t_rows = t_rows.copy()
            for r, i in enumerate(t_ids.tolist()):
                if i in at:
                    t_rows[r] = new[at[i]]
        states.append((t_rows, t_ids))
    wants = []
    for s_rows, s_ids in states:
        al = np.isin(s_ids, fset)
        wants.append([oracle.topk(s_rows[al], s_ids[al], q, k, 1e3, threads=oracle.max_threads()) for q in queries])

    def one_of(res, qi):
        return any(same(res, w[qi]) for w in wants)

    with Corpus(64, capacity_hint=len(ids)) as c:
        c.load(ids, rows)
        with c.view(fset) as v:
            done = threading.Event()
            seen = {"host": 0, "dev": 0}
            errors = []

            def host_searcher():
                while not done.is_set():
                    for qi, q in enumerate(queries):
                        r = v.search(q, k, 1e3)[0]
                        if not one_of(r, qi):
                            errors.append(("host", qi))
                    seen["host"] += 1

            def dev_searcher():
                s = torch.cuda.Stream()
                d_q = to_dev(queries)
                while not done.is_set():
                    out = DevOut(len(queries), k)
                    with torch.cuda.stream(s):
                        v.search_device(d_q.data_ptr(), len(queries), k, 1e3, *out.ptrs(), stream=s.cuda_stream)
                    s.synchronize()
                    for qi, r in enumerate(out.results()):
                        if not one_of(r, qi):
                            errors.append(("dev", qi))
                    seen["dev"] += 1

            ts = [threading.Thread(target=host_searcher), threading.Thread(target=dev_searcher)]
            for t in ts:
                t.start()
            try:
                for op, a, b in plan:
                    if op == "append":
                        c.append(a, b)
                    elif op == "remove":
                        c.remove(a)
                    else:
                        c.replace(a, b)
            finally:
                done.set()
                for t in ts:
                    t.join()
            assert not errors, errors[:5]
            assert seen["host"] and seen["dev"]
            for qi, q in enumerate(queries):                     # and the final state exactly
                assert same(v.search(q, k, 1e3)[0], wants[-1][qi])


# ---- sharded ----------------------------------------------------------------------------------------------------------------
def _sharded_view_check(devices):
    rng, rows, ids = table(77, 30_000, 256)
    fset = np.concatenate([ids[rng.random(len(ids)) < 0.05], ids[:40], [7, 11]])
    queries = np.concatenate([rows[rng.choice(len(rows), 4)], rows[np.isin(ids, fset)][:2]])
    with MultiDeviceCorpus(256, devices, capacity_hint=len(ids)) as m:
        m.load(ids, rows)
        v = m.view(fset)
        cur, t_rows, t_ids = np.unique(fset), rows.copy(), ids.copy()

        def state(msg):
            assert len(v) == int(np.isin(t_ids, cur).sum()), msg
            al = np.isin(t_ids, cur)
            for k, md in ((100, 1e3), (10, 1e3)):
                got = v.search(queries, k, md)
                want = m.search(queries, k, md, within=cur)
                for j, q in enumerate(queries):
                    assert same(got[j], fields(want[j])), f"{msg} k={k} q={j}"
                    if j < 2:
                        assert same(got[j], oracle.topk(t_rows[al], t_ids[al], q, k, md, threads=oracle.max_threads())), msg
            r = v.search(queries[0], 100, 1e3, after=[None])[0]
            assert same(r, fields(m.search(queries[0], 100, 1e3, within=cur)[0]))

        state("built")
        a_ids = np.array([7, 10 ** 9], np.int64)
        m.append(a_ids, queries[:2])
        t_rows, t_ids = np.concatenate([t_rows, queries[:2]]), np.concatenate([t_ids, a_ids])
        state("append")
        gone = np.concatenate([cur[:20], ids[100:200]])
        m.remove(gone)
        keep = ~np.isin(t_ids, gone)
        t_rows, t_ids = t_rows[keep], t_ids[keep]
        state("remove")
        pick = cur[30:60]
        new = clustered(rng, len(pick), 256)
        m.replace(pick, new)
        at = {int(i): j for j, i in enumerate(pick.tolist())}
        for r_, i in enumerate(t_ids.tolist()):
            if i in at:
                t_rows[r_] = new[at[i]]
        state("replace")
        add = t_ids[~np.isin(t_ids, cur)][:500]
        assert v.view_add(add) == len(add)
        cur = np.union1d(cur, add)
        state("view_add")
        drop = cur[::5]
        assert v.view_drop(drop) == int(np.isin(t_ids, drop).sum())
        cur = np.setdiff1d(cur, drop)
        state("view_drop")
        for call in (lambda: v.append(ids[:1], rows[:1]), lambda: v.remove(ids[:1]), lambda: v.load(ids[:1], rows[:1]),
                     lambda: v.replace(ids[:1], rows[:1]), lambda: v.fill_synthetic(10, 1), lambda: m.view_add(ids[:1])):
            with pytest.raises(nat.PbxError) as e:
                call()
            assert e.value.code == -1
        v.close()


@gpu
def test_sharded_view_three_shards_on_one_device():
    _sharded_view_check([0, 0, 0])


@gpu
def test_sharded_view_two_devices():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible")
    _sharded_view_check([0, 1])


@gpu
def test_view_exchange_two_processes():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29712", os.path.join(ROOT, "tools", "view_exchange_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "view_exchange_check OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]
