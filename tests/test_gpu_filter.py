"""Filtered searches (pbx_search_filtered and its twins, `within=` / `excluding=`): every path returns exactly what an
unfiltered search returns on a fresh corpus loaded with only the allowed rows -- ids, dist bit for bit, dot, norm2,
count -- which is also the oracle's top-k over those rows."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import Corpus, MultiDeviceCorpus, SearchResult

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def records(r):
    return sorted(zip(r.dist.view(np.uint32).tolist(), r.ids.tolist(), r.dot.tolist(), r.norm2.tolist()))


def same(a, b):
    """Ids and dist bit for bit in order, and the same (dist, id, dot, norm2) records.  Rows that share an image_id AND a
    dist (several rows with one id on the 999999 plateau) have no defined order among themselves -- a real table cannot
    hold them, image_id is its primary key -- so only their records are compared, not their order."""
    return (list(a.ids) == list(b.ids) and np.array_equal(a.dist.view(np.uint32), b.dist.view(np.uint32))
            and records(a) == records(b))


def same_oracle(res, want):
    o_ids, o_dist, o_dot, o_n2 = want
    return same(res, SearchResult(np.asarray(o_ids), np.asarray(o_dist, np.float32), np.asarray(o_dot), np.asarray(o_n2)))


def clustered(rng, n, d, spread=3, centres=30):
    cent = rng.integers(0, 256, size=(centres, d))
    return np.clip(cent[rng.integers(0, centres, n)] + rng.integers(-spread, spread + 1, size=(n, d)), 0, 255).astype(np.uint8)


def allowed_mask(ids, kw, fset):
    hit = np.isin(ids, fset)
    return hit if kw == "within" else ~hit


def reference(d, ids, rows, mask, cases):
    """{(queries id, k, md): unfiltered results} on a fresh corpus holding only the allowed rows (same nq, so the same path)."""
    with Corpus(d, capacity_hint=max(int(mask.sum()), 1)) as r:
        if mask.any():
            r.load(ids[mask], rows[mask])
        return {key: r.search(qs, k, md) for key, (qs, k, md) in cases.items()}


# ---- modes, sets, shapes, plateau, k above the allowed count, forced exact pass ---------------------------------------
@pytest.mark.parametrize("d", [8, 100, 256])
def test_filter_equals_a_corpus_of_the_allowed_rows(d):
    rng = np.random.default_rng(900 + d)
    n = 12_000
    rows = clustered(rng, n, d)
    rows[50:80] = rows[50]                              # plateau of identical rows, half of it in the sets below
    rows[n - 30:] = rows[50]
    ids = (rng.permutation(np.arange(1, n + 1)) * 3).astype(np.int64)
    ids[200:205] = ids[199]                             # one id on several rows
    sets = {
        "empty": np.array([], np.int64),
        "one": ids[[4321]],
        "1%": ids[rng.random(n) < 0.01],
        "50%": ids[rng.random(n) < 0.5],
        "99%": ids[rng.random(n) < 0.99],
        "absent": np.array([-5, 1, 2, 10**12], np.int64),            # ids are multiples of 3
        "plateau_half": np.concatenate([ids[50:65], ids[n - 15:], ids[199:200]]),
        "dups_unsorted": rng.permutation(np.concatenate([ids[1000:1100], ids[1000:1050], ids[199:201]])),
    }
    queries = np.concatenate([rows[[50, 5000]], rng.integers(0, 256, size=(2, d), dtype=np.uint8)])
    kmd = ((10, 1e3), (100, 1e3), (1000, 1e3), (100, 1e7), (100, 0.05))
    with Corpus(d, capacity_hint=n) as c:
        c.load(ids, rows)
        for slack in (0, 1):
            c.set_candidate_slack(slack)
            xp0 = c.stats().exact_passes
            for name, fset in sets.items():
                for kw in ("within", "excluding"):
                    mask = allowed_mask(ids, kw, fset)
                    wants = reference(d, ids, rows, mask, {(k, md): (queries, k, md) for k, md in kmd})
                    for k, md in kmd:
                        want = wants[(k, md)]
                        got = c.search(queries, k, md, **{kw: fset})                     # batched when the shape allows
                        assert all(same(g, w) for g, w in zip(got, want)), f"{name} {kw} d={d} slack={slack} k={k} md={md}"
                        for j in (0, 3):                                                  # the single-query path
                            one = c.search(queries[j], k, md, **{kw: fset})[0]
                            assert same(one, want[j]), f"single {name} {kw} d={d} slack={slack} k={k} md={md} q={j}"
                        if name == "empty" and kw == "within":
                            assert all(len(g.ids) == 0 for g in got)
                        if name == "empty" and kw == "excluding":
                            assert all(same(g, u) for g, u in zip(got, c.search(queries, k, md)))
                if slack == 0 and name in ("1%", "plateau_half"):
                    mask = allowed_mask(ids, "within", fset)
                    for q in queries[:2]:
                        assert same_oracle(c.search(q, 100, 1e7, within=fset)[0], oracle.topk(rows[mask], ids[mask], q, 100, 1e7, threads=4))
            if slack == 1:
                assert c.stats().exact_passes > xp0, "a candidate slack of 1 forced no exact pass"


# ---- the seeded single-query path and the batched path, dense and very selective sets --------------------------------
@pytest.fixture(scope="module")
def big():
    """400k x 64 synthetic rows (ids = row + 1): enough for prep_seed_kernel's sample (148 * 256 * 8 rows)."""
    n, d = 400_000, 64
    c = Corpus(d, capacity_hint=n)
    c.fill_synthetic(n, 11, 0)
    ids, rows = c.read_rows(0, n)
    yield c, ids, rows
    c.close()


def big_sets(ids):
    rng = np.random.default_rng(3)
    return {"dense": ids[rng.random(len(ids)) < 0.5],
            # ~40 allowed rows: the seed sample (148 x 256 rows) holds fewer than keep of them, no starting threshold
            "selective": ids[rng.choice(len(ids), 40, replace=False)],
            "selective_1k": ids[rng.choice(len(ids), 1000, replace=False)]}


def test_seeded_single_query_path(big):
    c, ids, rows = big
    d = rows.shape[1]
    queries = np.concatenate([rows[[7, 250_000]], np.random.default_rng(4).integers(0, 256, size=(2, d), dtype=np.uint8)])
    for name, fset in big_sets(ids).items():
        for kw in ("within", "excluding"):
            mask = allowed_mask(ids, kw, fset)
            for k in (100, 1000):
                want = reference(d, ids, rows, mask, {0: (queries[:1], k, 1e3)})[0][0]
                for j, q in enumerate(queries):
                    got = c.search(q, k, 1e3, **{kw: fset})[0]
                    if j == 0:
                        assert same(got, want), f"{name} {kw} k={k}"
                    if kw == "within" or j == 1:
                        assert same_oracle(got, oracle.topk(rows[mask], ids[mask], q, k, 1e3, threads=8)), f"{name} {kw} k={k} q={j}"


@pytest.mark.parametrize("seg", [None, "3"])
def test_batched_path(big, seg):
    c, ids, rows = big
    d = rows.shape[1]
    queries = np.concatenate([rows[[7, 250_000]], np.random.default_rng(5).integers(0, 256, size=(14, d), dtype=np.uint8)])
    old = os.environ.pop("PBX_BATCH_SEG_TILES", None)
    if seg:
        os.environ["PBX_BATCH_SEG_TILES"] = seg          # segmented main passes with cut-backs in between
    try:
        for name, fset in big_sets(ids).items():
            for kw in ("within", "excluding"):
                mask = allowed_mask(ids, kw, fset)
                want = reference(d, ids, rows, mask, {0: (queries, 100, 1e3)})[0]
                before = c.stats().batched_queries
                got = c.search(queries, 100, 1e3, **{kw: fset})
                assert c.stats().batched_queries == before + len(queries), "the tensor-core path did not run"
                assert all(same(g, w) for g, w in zip(got, want)), f"{name} {kw} seg={seg}"
                for j in (0, 5):
                    assert same_oracle(got[j], oracle.topk(rows[mask], ids[mask], queries[j], 100, 1e3, threads=8)), f"{name} {kw} q={j}"
    finally:
        os.environ.pop("PBX_BATCH_SEG_TILES", None)
        if old is not None:
            os.environ["PBX_BATCH_SEG_TILES"] = old


# ---- the filter follows ids, not positions -------------------------------------------------------------------------
def test_filter_after_remove_append_and_pending_appends():
    rng = np.random.default_rng(17)
    n, d = 20_000, 256
    rows = clustered(rng, n + 600, d)
    ids = np.arange(1, n + 601, dtype=np.int64) * 2
    fset = ids[rng.random(n + 600) < 0.2]
    queries = np.concatenate([rows[[10, 19_990, n + 5]], rng.integers(0, 256, size=(3, d), dtype=np.uint8)])
    with Corpus(d) as c:
        c.load(ids[:n], rows[:n])
        live = np.zeros(n + 600, bool)
        live[:n] = True
        gone = ids[:n][rng.random(n) < 0.3]
        c.remove(gone)                                    # survivors from the tail move into the holes
        live &= ~np.isin(ids, gone)
        c.append(ids[n:n + 500], rows[n:n + 500])
        live[n:n + 500] = True
        for i in range(n + 500, n + 600):                 # coalesced pending appends
            c.append(ids[i:i + 1], rows[i:i + 1])
        live[n + 500:] = True
        for kw in ("within", "excluding"):
            mask = live & allowed_mask(ids, kw, fset)
            want = reference(d, ids, rows, mask, {0: (queries, 100, 1e3)})[0]
            got = c.search(queries, 100, 1e3, **{kw: fset})
            assert all(same(g, w) for g, w in zip(got, want)), kw
            for j in (0, 2):
                assert same(c.search(queries[j], 100, 1e3, **{kw: fset})[0], want[j]), f"{kw} single q={j}"


# ---- device form --------------------------------------------------------------------------------------------------
def test_device_form_sorted_and_unsorted():
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(29)
    n, d, k = 30_000, 256, 100
    rows = clustered(rng, n, d)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    fset = np.unique(ids[rng.random(n) < 0.1])
    queries = np.concatenate([rows[[3]], rng.integers(0, 256, size=(7, d), dtype=np.uint8)])
    dev = torch.device("cuda", 0)
    with Corpus(d) as c:
        c.load(ids, rows)
        for nq in (1, 8):                                     # the single-query and the batched path
            d_q = torch.from_numpy(queries[:nq].copy()).to(dev)
            hits = torch.empty(nq * k * nat.HIT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
            cnt = torch.empty(nq, dtype=torch.int32, device=dev)
            for mode, kw in ((nat.PBX_FILTER_INCLUDE, "within"), (nat.PBX_FILTER_EXCLUDE, "excluding")):
                want = c.search(queries[:nq], k, 1e3, **{kw: fset})
                with_dups = np.sort(np.concatenate([fset, fset[:50]]))            # duplicates are allowed
                d_f = torch.from_numpy(with_dups).to(dev)
                stream = torch.cuda.current_stream().cuda_stream
                c.search_device_filtered(d_q.data_ptr(), nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), d_f.data_ptr(), d_f.numel(), mode, stream)
                torch.cuda.synchronize()
                h = hits.cpu().numpy().view(nat.HIT_DTYPE).reshape(nq, k)
                cn = cnt.cpu().numpy().astype(np.uint32)
                for i in range(nq):
                    assert cn[i] == len(want[i].ids)
                    assert list(h[i]["image_id"][:cn[i]]) == list(want[i].ids)
                    assert np.array_equal(h[i]["dist"][:cn[i]].view(np.uint32), want[i].dist.view(np.uint32))
                    assert np.array_equal(h[i]["dot"][:cn[i]], want[i].dot) and np.array_equal(h[i]["norm2"][:cn[i]], want[i].norm2)
                d_u = torch.from_numpy(with_dups[::-1].copy()).to(dev)               # descending: unsorted
                c.search_device_filtered(d_q.data_ptr(), nq, k, 1e3, hits.data_ptr(), cnt.data_ptr(), d_u.data_ptr(), d_u.numel(), mode, stream)
                torch.cuda.synchronize()
                assert (cnt.cpu().numpy().astype(np.uint32) == nat.PBX_COUNT_FILTER_UNSORTED).all(), f"mode {mode} nq {nq}"
                # the next search is unaffected
                assert all(same(g, w) for g, w in zip(c.search(queries[:nq], k, 1e3, **{kw: fset}), want))


# ---- sharded in one process -------------------------------------------------------------------------------------------
def _multi(devices):
    rng = np.random.default_rng(41)
    n, d = 40_000, 256
    rows = clustered(rng, n, d)
    rows[100:300] = rows[100]
    rows[n - 200:] = rows[100]
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 11
    queries = np.concatenate([rows[[100, 20_000]], rng.integers(0, 256, size=(10, d), dtype=np.uint8)])
    sets = [("within", np.concatenate([ids[rng.random(n) < 0.05], ids[150:250]])), ("excluding", ids[rng.random(n) < 0.5]),
            ("within", ids[[5]])]
    with Corpus(d) as one, MultiDeviceCorpus(d, devices) as mc:
        one.load(ids, rows)
        mc.load(ids, rows)
        for kw, fset in sets:
            for k, md, qs in ((100, 1e3, queries), (10, 1e3, queries[:1]), (500, 1e7, queries[:2])):
                got = mc.search(qs, k, md, **{kw: fset})
                want = one.search(qs, k, md, **{kw: fset})
                assert all(same(g, w) for g, w in zip(got, want)), f"{kw} k={k} md={md}"
                mask = allowed_mask(ids, kw, fset)
                assert same_oracle(got[0], oracle.topk(rows[mask], ids[mask], qs[0], k, md, threads=8))


def test_multi_device_corpus_on_one_gpu():
    _multi([0, 0, 0])


@pytest.mark.multigpu
def test_multi_device_corpus_on_two_gpus():
    _multi([0, 1])


# ---- one process per GPU ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_corpus_between_processes_sharing_one_gpu(world):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(29680 + world), os.path.join(ROOT, "tools", "filter_exchange_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "filter_exchange_check OK" in res.stdout, res.stdout[-3000:] + res.stderr[-3000:]


# ---- the Engine mirror -------------------------------------------------------------------------------------------
def test_engine_query_within_folder_matches_sql(tmp_path):
    from pixelbox_b200.engine import Engine, IndexedImage
    from tests import sqlite_oracle
    rng = np.random.default_rng(53)
    n, d = 3000, 64
    rows = clustered(rng, n, d)
    rows[10:40] = rows[10]                               # ties across the folders
    ids = np.arange(1, n + 1, dtype=np.int64)
    folders = ["/photos/a_b%c/", "/photos/axbyc/", "/photos/a_b%c2/"]     # % and _ are literal; a prefix of a name is not a folder
    path = str(tmp_path / "pbx.db")
    conn = sqlite_oracle.make_db(path, ids, rows)
    conn.executemany("UPDATE images SET path = ? WHERE id = ?",
                     [(f"{folders[int(i) % 3]}img{int(i)}.png", int(i)) for i in ids])
    conn.execute("DELETE FROM images WHERE id IN (10, 11, 12)")        # orphan hashes: in no folder
    conn.commit()
    eng = Engine.open(path)
    sql = sqlite_oracle.similarity_sql(100).replace("WHERE dist < ?", "WHERE dist < ? AND substr(images.path, 1, length(?)) = ?")
    try:
        for folder in ("/photos/a_b%c", "/photos/axbyc/", "/photos/nothing"):
            prefix = folder if folder.endswith("/") else folder + "/"
            for qi in (10, 500, 2999):
                for md in (1e3, 0.02):
                    eng.max_distance_from_query = md
                    eng.query_by_image_hash_within_folder(IndexedImage(visual_hash=bytes(rows[qi])), folder)
                    got = eng.get_query_results()
                    want = conn.execute(sql, (bytes(rows[qi]), md, prefix, prefix)).fetchall()
                    assert [g.id for g in got] == [w[0] for w in want], (folder, qi, md)
                    assert [g.distance_from_query for g in got] == [w[7] for w in want]
                    assert all(g.path.startswith(prefix) for g in got)
    finally:
        eng.close()
        conn.close()
