"""The batched-query (tensor-core) path against the oracle and against the single-query path:
identical ids, f32 distance bits and integer terms, for every row pitch it supports."""
import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import synth
from pixelbox_b200.corpus import Corpus
from tests import synth_oracle

pytestmark = pytest.mark.gpu


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def clustered(rng, n, d, ncent, noise):
    cent = rng.integers(0, 256, size=(ncent, d))
    x = cent[rng.integers(0, ncent, size=n)] + rng.integers(-noise, noise + 1, size=(n, d))
    return np.clip(x, 0, 255).astype(np.uint8)


def check(corpus, ids, queries, k, md, c, oracle_every=1):
    got = c.search(queries, k, md)
    for qi in range(0, len(queries), oracle_every):
        o_ids, o_dist, o_dot, o_n2 = oracle.topk(corpus, ids, queries[qi], k, md, threads=4)
        assert list(got[qi].ids) == list(o_ids), f"ids differ q={qi}"
        assert np.array_equal(bits(got[qi].dist), bits(o_dist)), f"dist bits differ q={qi}"
        assert np.array_equal(got[qi].dot, o_dot) and np.array_equal(got[qi].norm2, o_n2)
    return got


# row pitches with 128-byte K-chunks, and (new in round 2) 64- and 32-byte chunks: dim 64, 192, 320 / 32, 96, 100 (pitch 112 is
# not a multiple of 32 and must stay on the single-query path), 992
@pytest.mark.parametrize("d,n,nq", [(256, 60_000, 40), (256, 150_001, 700), (128, 50_000, 64), (512, 40_000, 300), (1024, 30_000, 130),
                                    (384, 40_000, 300), (640, 30_000, 130), (768, 30_000, 70), (896, 20_000, 33),
                                    (64, 120_000, 1024), (192, 50_000, 200), (320, 40_000, 129), (32, 100_000, 500), (96, 60_000, 257),
                                    (992, 20_000, 40), (250, 30_000, 64)])
def test_batched_equals_oracle_and_single_path(d, n, nq):
    rng = np.random.default_rng(d + nq)
    corpus = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    queries = rng.integers(0, 256, size=(nq, d), dtype=np.uint8)
    queries[: nq // 2] = np.clip(corpus[rng.integers(0, n, nq // 2)].astype(int) + rng.integers(-20, 21, size=(nq // 2, d)), 0, 255)
    with Corpus(d) as c:
        c.load(ids, corpus)
        before = c.stats().batched_queries
        batched = check(corpus, ids, queries, 100, 1e3, c, oracle_every=max(1, nq // 24))
        assert c.stats().batched_queries == before + nq, "the tensor-core path did not run"
        c.set_batch_min(0xFFFFFFFF)
        single = c.search(queries, 100, 1e3)
        assert c.stats().batched_queries == before + nq
        for a, b in zip(batched, single):
            assert list(a.ids) == list(b.ids) and np.array_equal(bits(a.dist), bits(b.dist))
            assert np.array_equal(a.dot, b.dot) and np.array_equal(a.norm2, b.norm2)


def test_batched_with_ties_filters_and_small_k():
    """Duplicates force the exact pass (tail-launched by the batched finalize kernel) for some queries only."""
    rng = np.random.default_rng(9)
    n, d = 80_000, 256
    corpus = clustered(rng, n, d, 2000, 1)
    corpus[1000:1600] = corpus[1000]                    # 600 identical rows
    ids = np.arange(1, n + 1, dtype=np.int64)
    queries = np.concatenate([corpus[[1000, 1001, 5, 77_777]], rng.integers(0, 256, size=(28, d), dtype=np.uint8)])
    with Corpus(d) as c:
        c.load(ids, corpus)
        for k, md in ((100, 1e3), (10, 1e3), (300, 0.05), (100, 1e7), (1000, 1e3), (2048, 1e3)):
            check(corpus, ids, queries, k, md, c)
        st = c.stats()
        # k = 1000 runs on the tensor cores with the large candidate buffers (16384 entries per query); k = 2048
        # (keep * 8 > 16384) is answered by the single-query loop
        assert st.batched_queries == 5 * len(queries) and st.exact_passes > 0


def test_batched_k1000_large_buffers_on_a_bigger_corpus():
    """keep = 1280: flood round of 20 tiles, candidate buffers of 16384 entries, cut back after the last round too."""
    n, d, nq, k = 600_000, 256, 40, 1000
    corpus = synth.synth_rows(21, 0, n, d)
    ids = np.arange(1, n + 1, dtype=np.int64)
    queries = synth.synth_queries(22, nq, d, n, 21)
    with Corpus(d) as c:
        c.load(ids, corpus)
        before = c.stats().batched_queries
        got = c.search(queries, k)
        assert c.stats().batched_queries == before + nq, "the tensor-core path did not run"
        for qi in range(0, nq, 7):
            o_ids, o_dist, o_dot, o_n2 = oracle.topk(corpus, ids, queries[qi], k, 1e3, threads=oracle.max_threads())
            assert list(got[qi].ids) == list(o_ids), qi
            assert np.array_equal(np.asarray(got[qi].dist).view(np.uint32), o_dist.view(np.uint32)), qi
            assert np.array_equal(got[qi].dot, o_dot) and np.array_equal(got[qi].norm2, o_n2)


@pytest.mark.parametrize("d,n", [(64, 40_000), (256, 30_000), (32, 50_000), (1024, 8_000)])
def test_batched_bound_with_wild_norm_spread_and_negative_thresholds(d, n):
    """The epilogue tests max(32 raw scores) against ONE bound per query and 32-row block, built from the block's norm
    range, its largest row term and the query's threshold (batch_bound_t4 / batch_bound_cq).  A bound that is too tight
    loses a true neighbour silently (the certificate only sees candidates that were found), so: blocks that mix rows of
    almost no norm (bytes 127 / 128), of maximal norm (bytes 0 / 255) and ordinary rows; queries of all three kinds and
    their complements (all cosines negative: negative thresholds); every query checked against the oracle."""
    rng = np.random.default_rng(1000 + d)
    kind = rng.integers(0, 4, size=n)
    corpus = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    tiny = rng.integers(127, 129, size=(n, d), dtype=np.uint8)
    huge = (rng.integers(0, 2, size=(n, d), dtype=np.uint8) * 255).astype(np.uint8)
    dark = rng.integers(0, 40, size=(n, d), dtype=np.uint8)             # large norm, large negative row term
    corpus[kind == 1] = tiny[kind == 1]
    corpus[kind == 2] = huge[kind == 2]
    corpus[kind == 3] = dark[kind == 3]
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    base = corpus[rng.integers(0, n, 24)].astype(int)
    near = np.clip(base + rng.integers(-3, 4, size=base.shape), 0, 255).astype(np.uint8)
    queries = np.concatenate([near, (255 - near).astype(np.uint8), rng.integers(0, 256, size=(8, d), dtype=np.uint8),
                              np.full((1, d), 128, np.uint8), np.full((1, d), 0, np.uint8), np.full((1, d), 255, np.uint8)])
    with Corpus(d) as c:
        c.load(ids, corpus)
        for k, md in ((100, 1e7), (10, 1e3), (300, 1e7)):
            before = c.stats().batched_queries
            check(corpus, ids, queries, k, md, c)
            # (k = 300 needs 562 sampled 32-row blocks for its seed: the smallest corpus here answers it query by query)
            assert k > 100 or c.stats().batched_queries == before + len(queries), "the tensor-core path did not run"


def test_full_size_10m_batch_of_1024_properties():
    """BASELINE configs[2] at full size (10M x 256, 1024 queries, top-100) through the tensor-core path, every query checked in
    full against the complete reference of the synthetic corpus (tests/synth_oracle.py): ids, order, distance bits, integer
    terms.  Planted self-matches lead with the reference's self-distance; 16 of the queries through the single-query path
    give the same answers."""
    n, d, k, nq, seed = 10_000_000, 256, 100, 1024, 42
    with Corpus(d, capacity_hint=n) as c:
        c.fill_synthetic(n, seed, 0)
        queries = synth.synth_queries(43, nq, d, n, seed)
        probes = {0: 17, 500: 5_000_000, 1023: n - 1}
        for qi, row in probes.items():
            queries[qi] = synth.synth_rows(seed, row, 1, d)[0]
        before = c.stats().batched_queries
        res = c.search(queries, k)
        assert c.stats().batched_queries == before + nq, "the tensor-core path did not run"
        want = synth_oracle.SynthReference(n, seed, d, 0, device="cuda").topk(queries, k)
        for qi in range(nq):
            r, (o_ids, o_dist, o_dot, o_n2) = res[qi], want[qi]
            assert len(r.ids) == k
            assert list(r.ids) == list(o_ids) and np.array_equal(bits(r.dist), bits(o_dist)), f"q{qi}: differs from the reference"
            assert np.array_equal(r.dot, o_dot) and np.array_equal(r.norm2, o_n2)
            if qi in probes:
                assert r.ids[0] == probes[qi] + 1
                assert bits(r.dist[0]) == bits(oracle.cosine_distance(queries[qi], queries[qi]))
        rng = np.random.default_rng(8)
        checked = sorted(set(probes) | set(int(x) for x in rng.integers(0, nq, 13)))
        c.set_batch_min(0xFFFFFFFF)
        single = c.search(queries[checked], k)
        for qi, b in zip(checked, single):
            a = res[qi]
            assert list(a.ids) == list(b.ids) and np.array_equal(bits(a.dist), bits(b.dist)), f"q{qi}: single-query path differs"
        assert c.stats().batched_queries == before + nq


def test_main_pass_in_segments_gives_the_same_answers(monkeypatch):
    """Long shards with large candidate sets run the main pass in segments with a cut-back of the candidate buffers in
    between (a buffer that overflows costs its query an exact pass).  Forced here on a small shard (PBX_BATCH_SEG_TILES):
    thresholds and candidates carry over from segment to segment, the answers are the oracle's."""
    monkeypatch.setenv("PBX_BATCH_SEG_TILES", "37")
    n, d, nq = 150_000, 256, 48
    rng = np.random.default_rng(77)
    corpus = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    queries = rng.integers(0, 256, size=(nq, d), dtype=np.uint8)
    queries[:16] = corpus[rng.integers(0, n, 16)]
    with Corpus(d) as c:
        c.load(ids, corpus)
        for k in (100, 400):
            before = c.stats().batched_queries
            check(corpus, ids, queries, k, 1e3, c, oracle_every=3)
            assert c.stats().batched_queries == before + nq, "the tensor-core path did not run"
