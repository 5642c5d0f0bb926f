"""Parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle and the
committed golden fixtures.  Bit-exact everywhere: ids, f32 distance bits, int32 dot / norm2."""
import json
import os

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200 import synth
from pixelbox_b200.corpus import Corpus, cosine_distance_pairs
from tests import synth_oracle

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def assert_same(res, want, ctx=""):
    o_ids, o_dist, o_dot, o_n2 = want
    assert list(res.ids) == list(o_ids), f"ids differ {ctx}"
    assert np.array_equal(bits(res.dist), bits(o_dist)), f"dist bits differ {ctx}"
    assert np.array_equal(res.dot, o_dot), f"dot differs {ctx}"
    assert np.array_equal(res.norm2, o_n2), f"norm2 differs {ctx}"


def check_against_oracle(corpus, ids, queries, ks=(10, 100), mds=(1e3,), slack=None, ctx=""):
    n, d = corpus.shape
    with Corpus(d) as c:
        c.load(ids, corpus)
        assert len(c) == n
        if slack is not None:
            c.set_candidate_slack(slack)
        for k in ks:
            for md in mds:
                want = [oracle.topk(corpus, ids, q, k, md) for q in queries]
                # every call both ways: looping over the single-query scan, and whatever the default dispatch picks
                # (the tensor-core batched path from 2 queries on, where the shape allows it)
                for batch_min, mode in ((0xFFFFFFFF, "single"), (0, "default")):
                    c.set_batch_min(batch_min)
                    got = c.search(queries, k, md)
                    for qi in range(len(queries)):
                        assert_same(got[qi], want[qi], f"{ctx} {mode} n={n} d={d} k={k} md={md} q={qi}")
        return c.stats()


def clustered(rng, n, d, ncent, noise):
    cent = rng.integers(0, 256, size=(ncent, d))
    x = cent[rng.integers(0, ncent, size=n)] + rng.integers(-noise, noise + 1, size=(n, d))
    return np.clip(x, 0, 255).astype(np.uint8)


def test_upstream_kat_on_gpu():
    # src/engine.rs:703-708 through the GPU pair kernel
    a = np.array([[255, 0], [0, 255], [255, 0]], np.uint8)
    b = np.array([[255, 0], [0, 255], [0, 255]], np.uint8)
    dist, dot, na, nb = cosine_distance_pairs(a, b)
    assert dist[0] < 1e-6 and dist[1] < 1e-6 and dist[2] > 2.0
    assert dist[2] == np.float32(999999.0)
    assert list(dot) == [2 * 255 * 255, 2 * 255 * 255, -2 * 255 * 255]


def test_golden_cosine_pairs():
    with open(os.path.join(GOLDEN, "cosine_pairs.json")) as f:
        pairs = [p for p in json.load(f) if len(p["a"]) == len(p["b"]) and len(p["a"]) > 0]
    by_len = {}
    for p in pairs:
        by_len.setdefault(len(p["a"]) // 2, []).append(p)
    assert len(by_len) >= 8
    for d, ps in by_len.items():
        a = np.stack([np.frombuffer(bytes.fromhex(p["a"]), np.uint8) for p in ps])
        b = np.stack([np.frombuffer(bytes.fromhex(p["b"]), np.uint8) for p in ps])
        dist, dot, na, nb = cosine_distance_pairs(a, b)
        assert [int(x) for x in bits(dist)] == [p["dist_bits"] for p in ps], d
        assert list(dot) == [p["dot"] for p in ps]
        assert list(na) == [p["norm2_a"] for p in ps]
        assert list(nb) == [p["norm2_b"] for p in ps]


def test_golden_topk_fixture():
    z = np.load(os.path.join(GOLDEN, "topk_small.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    assert len(names) == 6
    for name in names:
        corpus, ids, queries = z[f"{name}/corpus"], z[f"{name}/ids"], z[f"{name}/queries"]
        with Corpus(corpus.shape[1]) as c:
            c.load(ids, corpus)
            for k, md in ((10, 1e3), (50, 1e3), (100, 1e3), (100, 0.5), (100, 1e7)):
                got = c.search(queries, k, md)
                for qi in range(len(queries)):
                    key = f"{name}/q{qi}/k{k}/md{md:g}"
                    assert list(got[qi].ids) == list(z[key + "/ids"]), key
                    assert np.array_equal(bits(got[qi].dist), z[key + "/dist_bits"]), key
                    assert np.array_equal(got[qi].dot, z[key + "/dot"]), key
                    assert np.array_equal(got[qi].norm2, z[key + "/norm2"]), key


@pytest.mark.parametrize("d", [1, 3, 8, 13, 16, 24, 32, 48, 64, 80, 96, 100, 128, 160, 192, 200, 256, 272, 320, 384, 512, 640, 768, 1000,
                               1024, 1280, 1536, 1792, 2048, 2100, 2560, 3072, 4000, 4096])
def test_random_corpus_every_row_shape(d):
    """Every kernel shape: compile-time layouts (pitch = 1, 3, 5, 6 or 8 times a power of two chunks: 16..4096 bytes)
    and the ragged layouts for everything else (e.g. pitches 112, 208, 272, 1008, 1792, 2112, 4000), with ragged n."""
    rng = np.random.default_rng(1000 + d)
    for n in (1, 33, 1500, 4097):
        corpus = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
        ids = np.sort(rng.choice(np.arange(1, 20 * n + 2), size=n, replace=False)).astype(np.int64)
        queries = np.stack([corpus[n // 2], rng.integers(0, 256, d, dtype=np.uint8),
                            np.clip(corpus[0].astype(int) + rng.integers(-5, 6, d), 0, 255).astype(np.uint8)])
        check_against_oracle(corpus, ids, queries, ks=(7, 100), mds=(1e3, 0.9))


@pytest.mark.parametrize("d", [8, 64, 100, 256, 384, 1000, 1280])
def test_heavy_ties_need_the_exact_pass(d):
    """More identical rows than candidates: order must be by image_id, ids deliberately unsorted
    with respect to row order (SQLite scans by rowid, we scan by load order)."""
    rng = np.random.default_rng(77 + d)
    n = 20000
    corpus = clustered(rng, n, d, 6, 0)               # 6 distinct vectors only
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    queries = np.stack([corpus[5], corpus[11], rng.integers(0, 256, d, dtype=np.uint8)])
    st = check_against_oracle(corpus, ids, queries, ks=(100, 1000), mds=(1e3,))
    assert st.exact_passes > 0


@pytest.mark.parametrize("d", [16, 256])
def test_forced_exact_pass_changes_nothing(d):
    rng = np.random.default_rng(5 + d)
    n = 30000
    corpus = clustered(rng, n, d, 300, 2)
    ids = np.arange(1, n + 1, dtype=np.int64)
    queries = np.stack([corpus[17], corpus[29999], rng.integers(0, 256, d, dtype=np.uint8)])
    st = check_against_oracle(corpus, ids, queries, ks=(50,), mds=(1e3, 0.02), slack=1)
    assert st.exact_passes >= 3
    st2 = check_against_oracle(corpus, ids, queries, ks=(50,), mds=(1e3, 0.02))
    assert st2.exact_passes <= st.exact_passes


def test_plateau_rows_are_ordered_by_id():
    """max_dist above 999999 admits the cos <= 1e-6 plateau (src/engine.rs:587): every such row has
    dist == 999999.0 exactly and SQLite orders them by image_id."""
    rng = np.random.default_rng(8)
    for n, d, k in ((150, 8, 100), (6000, 64, 100), (6000, 64, 2000)):
        corpus = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
        ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
        q = rng.integers(0, 256, d, dtype=np.uint8)
        anti = (255 - q).astype(np.uint8)              # the query's antipode: every row with positive cos to it is on the plateau
        check_against_oracle(corpus, ids, np.stack([q, anti]), ks=(k,), mds=(1e7, 999999.0, 999999.5))
    # a corpus that is entirely on the plateau
    corpus = np.tile(anti, (5000, 1))
    corpus[:, 0] = rng.integers(0, 4, 5000)
    check_against_oracle(corpus, rng.permutation(np.arange(10, 5010)).astype(np.int64), np.stack([q]), ks=(100,), mds=(1e7, 1e3))


def test_filter_is_strict_less_than_in_f64():
    rng = np.random.default_rng(3)
    corpus = clustered(rng, 3000, 32, 20, 3)
    ids = np.arange(1, 3001, dtype=np.int64)
    q = corpus[100]
    dists = np.sort(np.unique(oracle.all_distances(corpus, q)))
    mids = [float(dists[5]), float(np.nextafter(dists[5], np.float32(np.inf))), float(dists[40]), 0.0, -1.0, float(dists[0])]
    check_against_oracle(corpus, ids, np.stack([q]), ks=(100,), mds=mids)


def test_append_equals_load_and_ids_are_opaque():
    rng = np.random.default_rng(21)
    n, d = 7000, 64
    corpus = clustered(rng, n, d, 50, 4)
    ids = (rng.permutation(n).astype(np.int64) - 3000) * 1_000_003      # negative and huge ids
    q = np.stack([corpus[3], rng.integers(0, 256, d, dtype=np.uint8)])
    with Corpus(d, capacity_hint=10) as c:
        for lo in range(0, n, 999):                                     # grows several times
            c.append(ids[lo:lo + 999], corpus[lo:lo + 999])
            assert len(c) == min(n, lo + 999)
        got = c.search(q, 100, 1e3)
        for qi in range(2):
            assert_same(got[qi], oracle.topk(corpus, ids, q[qi], 100, 1e3))
        r_ids, r_rows = c.read_rows(0, n)
        assert np.array_equal(r_ids, ids) and np.array_equal(r_rows, corpus)
        # prefix semantics: a later load replaces everything
        c.load(ids[:100], corpus[:100])
        assert len(c) == 100
        assert_same(c.search(q[:1], 100, 1e3)[0], oracle.topk(corpus[:100], ids[:100], q[0], 100, 1e3))


def test_empty_corpus_and_argument_errors():
    with Corpus(16) as c:
        res = c.search(np.zeros((2, 16), np.uint8), 10)
        assert len(res) == 2 and all(len(r.ids) == 0 for r in res)
        with pytest.raises(nat.PbxError) as e1:
            c.search(np.zeros((1, 15), np.uint8), 10)
        assert e1.value.code == -2
        with pytest.raises(nat.PbxError) as e2:
            c.search(np.zeros((1, 16), np.uint8), 0)
        assert e2.value.code == -1
        with pytest.raises(nat.PbxError) as e3:
            c.search(np.zeros((1, 16), np.uint8), nat.PBX_MAX_K + 1)
        assert e3.value.code == -7
        with pytest.raises(nat.PbxError):
            c.append([1, 2], np.zeros((2, 17), np.uint8))


def test_synthetic_fill_matches_host_definition():
    for d, n, first in ((256, 5000, 0), (64, 3000, 1 << 33), (13, 777, 5), (1024, 600, 123456789)):
        with Corpus(d) as c:
            c.fill_synthetic(n, 42, first)
            ids, rows = c.read_rows(0, n)
            assert np.array_equal(rows, synth.synth_rows(42, first, n, d))
            assert np.array_equal(ids, np.arange(first + 1, first + n + 1, dtype=np.int64))
            q = synth.synth_queries(7, 4, d, n, 42)
            got = c.search(q, 50)
            for qi in range(4):
                assert_same(got[qi], oracle.topk(rows, ids, q[qi], 50, 1e3))


def test_batch_equals_single_and_order_of_queries():
    rng = np.random.default_rng(99)
    corpus = rng.integers(0, 256, size=(9000, 256), dtype=np.uint8)
    ids = np.arange(1, 9001, dtype=np.int64)
    queries = rng.integers(0, 256, size=(37, 256), dtype=np.uint8)
    with Corpus(256) as c:
        c.load(ids, corpus)
        batch = c.search(queries, 20)
        for qi in (0, 5, 36):
            single = c.search(queries[qi], 20)[0]
            assert list(single.ids) == list(batch[qi].ids)
            assert_same(batch[qi], oracle.topk(corpus, ids, queries[qi], 20, 1e3))
        hits, cnt = c.search_hits(queries, 20)
        assert hits.shape == (37, 20) and all(cnt == 20)
        assert np.array_equal(hits["image_id"][5], batch[5].ids)


def test_device_resident_path_with_torch_buffers():
    import torch
    rng = np.random.default_rng(123)
    corpus = rng.integers(0, 256, size=(20000, 64), dtype=np.uint8)
    ids = np.arange(1, 20001, dtype=np.int64)
    queries = rng.integers(0, 256, size=(5, 64), dtype=np.uint8)
    k = 30
    with Corpus(64) as c:
        c.load(ids, corpus)
        dq = torch.from_numpy(queries).cuda()
        dh = torch.zeros(5 * k * 24, dtype=torch.uint8, device="cuda")
        dc = torch.zeros(5, dtype=torch.int32, device="cuda")
        s = torch.cuda.current_stream()
        c.search_device(dq.data_ptr(), 5, k, 1e3, dh.data_ptr(), dc.data_ptr(), s.cuda_stream)
        s.synchronize()
        hits = dh.cpu().numpy().view(nat.HIT_DTYPE).reshape(5, k)
        cnt = dc.cpu().numpy()
        for qi in range(5):
            o_ids, o_dist, _, _ = oracle.topk(corpus, ids, queries[qi], k, 1e3)
            assert cnt[qi] == len(o_ids)
            assert np.array_equal(hits[qi]["image_id"][:cnt[qi]], o_ids)
            assert np.array_equal(bits(hits[qi]["dist"][:cnt[qi]]), bits(o_dist))


def test_full_size_10m_properties():
    """BASELINE config 2 (10M x 256, top-100), every answer checked in full against the complete reference of the synthetic
    corpus (tests/synth_oracle.py); the planted self-matches lead with the reference's self-distance."""
    n, d, k, seed = 10_000_000, 256, 100, 42
    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed, 0)
        probe_rows = [0, 1234567, n - 1]
        queries = np.concatenate([synth.synth_rows(seed, r, 1, d) for r in probe_rows] + [synth.synth_queries(11, 6, d, n, seed)])
        res = c.search(queries, k)
        want = synth_oracle.SynthReference(n, seed, d, 0, device="cuda").topk(queries, k)
        for qi, r in enumerate(res):
            assert len(r.ids) == k
            assert_same(r, want[qi], f"q{qi} (complete reference)")
            if qi < len(probe_rows):
                assert r.ids[0] == probe_rows[qi] + 1
                assert bits(r.dist[0]) == bits(oracle.cosine_distance(queries[qi], queries[qi]))
        st = c.stats()
        assert st.rows == n and st.exact_passes == 0


def test_async_back_to_back_with_forced_exact_passes():
    """Queries enqueued back to back on one stream, each needing the exact pass (device-side tail launch):
    kernels of consecutive queries overlap through programmatic dependent launch and share scratch, so any
    ordering hole shows up as a wrong list."""
    import torch
    rng = np.random.default_rng(321)
    n, d, k = 300_000, 64, 40
    corpus = clustered(rng, n, d, 500, 1)
    ids = np.arange(1, n + 1, dtype=np.int64)
    nq = 24
    queries = np.stack([corpus[int(rng.integers(0, n))] for _ in range(nq)])
    with Corpus(d) as c:
        c.load(ids, corpus)
        for slack in (1, 0):                     # 1 forces the exact pass, 0 = default
            c.set_candidate_slack(slack)
            dq = torch.from_numpy(queries).cuda()
            dh = torch.zeros(nq * k * 24, dtype=torch.uint8, device="cuda")
            dc = torch.zeros(nq, dtype=torch.int32, device="cuda")
            s = torch.cuda.Stream()
            torch.cuda.synchronize()
            for rep in range(3):
                for qi in range(nq):
                    c.search_device(dq.data_ptr() + qi * d, 1, k, 1e3, dh.data_ptr() + qi * k * 24, dc.data_ptr() + 4 * qi, s.cuda_stream)
            s.synchronize()
            hits = dh.cpu().numpy().view(nat.HIT_DTYPE).reshape(nq, k)
            cnt = dc.cpu().numpy()
            for qi in range(nq):
                o_ids, o_dist, o_dot, _ = oracle.topk(corpus, ids, queries[qi], k, 1e3, threads=4)
                assert cnt[qi] == len(o_ids)
                assert np.array_equal(hits[qi]["image_id"][:cnt[qi]], o_ids), (slack, qi)
                assert np.array_equal(bits(hits[qi]["dist"][:cnt[qi]]), bits(o_dist))
                assert np.array_equal(hits[qi]["dot"][:cnt[qi]], o_dot)
        assert c.stats().exact_passes >= 3 * nq


def test_search_concurrent_with_append_sees_a_committed_prefix():
    """The writer thread of Engine::start_indexing (src/engine.rs:186-203) appends while the UI thread searches
    (src/ui/search.rs:22): every answer must be the reference's answer over some committed prefix of the rows."""
    import threading
    rng = np.random.default_rng(2024)
    n, d, k, block = 60_000, 64, 25, 2_000
    corpus = clustered(rng, n, d, 400, 3)
    ids = np.arange(1, n + 1, dtype=np.int64)
    queries = [corpus[int(rng.integers(0, n))] for _ in range(6)]
    with Corpus(d, capacity_hint=block) as c:           # small hint: the buffers are re-allocated many times
        c.append(ids[:block], corpus[:block])
        errors, seen = [], []

        def writer():
            try:
                for lo in range(block, n, block):
                    c.append(ids[lo:lo + block], corpus[lo:lo + block])
            except Exception as e:                      # pragma: no cover
                errors.append(e)

        t = threading.Thread(target=writer)
        t.start()
        while t.is_alive() or len(seen) < 12:
            q = queries[len(seen) % len(queries)]
            n0 = len(c)
            r = c.search(q, k)[0]
            n1 = len(c)
            seen.append((q, n0, n1, r))
            if len(seen) > 400:
                break
        t.join()
        assert not errors
        assert len(c) == n
        prefixes = set()
        for q, n0, n1, r in seen:
            ok = False
            for m in range(n0, n1 + 1, block):
                o_ids, o_dist, _, _ = oracle.topk(corpus[:m], ids[:m], q, k, 1e3, threads=4)
                if list(r.ids) == list(o_ids) and np.array_equal(bits(r.dist), bits(o_dist)):
                    ok = True
                    prefixes.add(m)
                    break
            assert ok, f"answer matches no committed prefix in [{n0}, {n1}]"
        assert len(prefixes) >= 1


@pytest.mark.parametrize("n_shards,k,nq", [(2, 100, 3), (8, 100, 5), (8, 1000, 2), (40, 100, 2), (64, 2048, 1), (3, 1, 4)])
def test_device_merge_equals_host_merge(n_shards, k, nq):
    """pbx_merge_hits_device (shared-memory staged keys when n_shards*k <= 8192, L2 probes above) against
    pbx_merge_hits: ties in dist across shards, duplicate (dist, id) pairs, short and empty lists, counts
    passed explicitly and implied by +inf tails."""
    import torch
    from pixelbox_b200.corpus import merge_hits
    rng = np.random.default_rng(n_shards * 1000 + k)
    gathered = np.zeros((n_shards, nq, k), nat.HIT_DTYPE)
    counts = np.zeros((n_shards, nq), np.uint32)
    for s in range(n_shards):
        for q in range(nq):
            c = int(rng.integers(0, k + 1)) if (s + q) % 3 else k
            if s == 1 and q == 0:
                c = 0
            dist = np.sort(rng.integers(0, 40, size=c).astype(np.float32) * 0.125 - 0.25)        # many ties, some negative
            ids = rng.integers(1, 50, size=c).astype(np.int64)
            order = np.lexsort((ids, dist))
            h = gathered[s, q]
            h["dist"][:c], h["image_id"][:c] = dist[order], ids[order]
            h["dot"][:c] = rng.integers(-1000, 1000, size=c)
            h["norm2"][:c] = s
            h["dist"][c:], h["image_id"][c:] = np.inf, np.iinfo(np.int64).max
            counts[s, q] = c
    want_hits, want_cnt = merge_hits(gathered, counts, k)
    d_g = torch.from_numpy(gathered.view(np.uint8).reshape(-1)).cuda()
    d_c = torch.from_numpy(counts.astype(np.int32).reshape(-1)).cuda()
    for with_counts in (True, False):
        d_out = torch.zeros(nq * k * 24, dtype=torch.uint8, device="cuda")
        d_cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")
        nat.check(nat.lib().pbx_merge_hits_device(0, d_g.data_ptr(), d_c.data_ptr() if with_counts else None, n_shards, nq, k,
                                                  d_out.data_ptr(), d_cnt.data_ptr(), torch.cuda.current_stream().cuda_stream or 1))
        torch.cuda.synchronize()
        got = d_out.cpu().numpy().view(nat.HIT_DTYPE).reshape(nq, k)
        got_cnt = d_cnt.cpu().numpy().astype(np.uint32)
        assert np.array_equal(got_cnt, want_cnt)
        for q in range(nq):
            n = int(want_cnt[q])
            for f in ("image_id", "dot"):
                assert np.array_equal(got[q][f][:n], want_hits[q][f][:n]), (f, q, with_counts)
            assert np.array_equal(bits(got[q]["dist"][:n]), bits(want_hits[q]["dist"][:n]))
