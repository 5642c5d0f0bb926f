"""Shards at full scale, every answer checked in full against the complete reference of synthetic corpora
(tests/synth_oracle.py): ids in order, dist bits, dot, norm2 and the count.

Row indices are 32-bit unsigned throughout the kernels (candidate keys, the removal's hole and source lists, replace's
pairs, a view's gather list, the mark bitmaps), and the batched path hands over to the single-query loop above
kBatchMaxRows rows because TMA row coordinates are signed 32-bit.  A signed or truncated index anywhere would lose or
alias rows past 2^31 and give plausible wrong answers; only shards that large can show it.  Three tiers, each a class
with its own corpus, never two resident at once:

* 100M x 256 (27.3 GB): every search path at k up to PBX_MAX_K, 1024-query batches (k = 1000 runs the main pass in
  25M-row segments), filters, pages past PBX_MAX_K, forced exact passes, then removal and replacement;
* dim 32 over 2^31 + 2^20 rows (104.2 GB): across 2^31 and the batched path's hand-over in both directions;
* dim 8 over PBX_MAX_ROWS rows (139.6 GB), ids past 2^32: the top of the range, and appends refused at the limit.
"""
import gc
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200 import synth
from pixelbox_b200.corpus import Corpus
from tests import synth_oracle

pytestmark = pytest.mark.gpu

K_BATCH_MAX_ROWS = 0x7FFFF000        # api.cu: rows the batched path can address
PBX_MAX_ROWS = 0xFFFFF000
PBX_E_CAPACITY = -6
REF_CHUNK = 2 << 30                  # float64 scratch of one reference chunk


def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def same(res, want, what):
    w_ids, w_dist, w_dot, w_n2 = want
    assert len(res.ids) == len(w_ids), f"{what}: {len(res.ids)} rows, the reference has {len(w_ids)}"
    assert list(res.ids) == list(w_ids), f"{what}: ids differ"
    assert np.array_equal(bits(res.dist), bits(w_dist)), f"{what}: dist bits differ"
    assert np.array_equal(res.dot, w_dot) and np.array_equal(res.norm2, w_n2), f"{what}: dot / norm2 differ"


def cut(want, lo, hi):
    """Rows [lo, hi) of a reference answer: the prefix of a deep top-K is the top-k, a slice of it is a page."""
    return tuple(a[lo:hi] for a in want)


def error_code(fn):
    try:
        fn()
    except nat.PbxError as e:
        return e.code
    return None


def sample(rng, lo, hi, count):
    """`count` distinct integers of [lo, hi), in random order."""
    out = np.zeros(0, np.int64)
    while out.size < count:
        out = np.unique(np.concatenate([out, rng.integers(lo, hi, count + count // 4 + 16)]))
    return rng.permutation(out)[:count]


def shard_bytes(n, dim):
    pitch = (dim + 15) // 16 * 16
    return n * (pitch + 4 + 4 + 8) + n // 32 * 16      # rows, inv_norm, row_sum, ids, block metadata


def open_tier(n, dim, seed, first_row=0):
    """The tier's corpus, filled on the device, and its reference.  Skips when the GPU cannot hold the shard, three
    reference chunks and 8 GB; the 8 GB also cover what the reference needs beyond its chunks (products of the largest
    batches, sort buffers of torch.topk)."""
    import torch
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    need = shard_bytes(n, dim) + 3 * REF_CHUNK
    if free < need + 8e9:
        pytest.skip(f"needs {need / 1e9:.1f} GB (shard and three reference chunks) + 8 GB free on the GPU; "
                    f"{free / 1e9:.1f} GB are free")
    c = Corpus(dim, capacity_hint=n)
    c.fill_synthetic(n, seed, first_row)
    ref = synth_oracle.SynthReference(n, seed, dim, first_row, device="cuda", chunk_bytes=REF_CHUNK)
    return SimpleNamespace(c=c, ref=ref, n=n, dim=dim, seed=seed, first_row=first_row, cache={})


def close_tier(t):
    import torch
    t.c.close()
    t.cache.clear()
    t.ref = None
    gc.collect()
    torch.cuda.empty_cache()


def cached(t, key, fn):
    if key not in t.cache:
        t.cache[key] = fn()
    return t.cache[key]


def self_match(res, t, row, what):
    """A query equal to local row `row` finds that row first, at the reference's self-distance."""
    q = t.ref.row_bytes([t.first_row + row + 1])[0]
    assert res.ids[0] == t.first_row + row + 1, f"{what}: row {row} does not lead its own result"
    assert bits(res.dist[0]) == bits(oracle.cosine_distance(q, q)), f"{what}: self-distance"


# ---------------------------------------------------------------------------------------------------------------------
# Tier 1: 100M x 256, everything checked in full
# ---------------------------------------------------------------------------------------------------------------------
T1_N, T1_DIM, T1_SEED = 100_000_000, 256, 2024
T1_PROBES = [0, 2**26 + 3, T1_N - 1]


@pytest.fixture(scope="class")
def t1():
    t = open_tier(T1_N, T1_DIM, T1_SEED)
    q = synth.synth_queries(91, 1024, T1_DIM, T1_N, T1_SEED)
    q[:3] = synth.synth_rows(T1_SEED, 0, 1, T1_DIM)[0], synth.synth_rows(T1_SEED, 2**26 + 3, 1, T1_DIM)[0], \
        synth.synth_rows(T1_SEED, T1_N - 1, 1, T1_DIM)[0]
    t.q1024 = q
    t.q16 = np.ascontiguousarray(q[:16])
    yield t
    close_tier(t)


class TestShard100Mx256:
    def deep(self, t):
        """The first 3000 rows of the 16 single-path queries: top-k for every k checked, and pages past PBX_MAX_K."""
        return cached(t, "deep", lambda: t.ref.topk(t.q16, 3000))

    def test_single_path_every_k(self, t1):
        c, want = t1.c, self.deep(t1)
        before = c.stats().batched_queries
        for k in (1, 10, 100, 1000, 2048):
            for qi in range(16):
                res = c.search(t1.q16[qi], k)[0]
                same(res, cut(want[qi], 0, k), f"single k={k} q{qi}")
                if qi < len(T1_PROBES):
                    self_match(res, t1, T1_PROBES[qi], f"single k={k} q{qi}")
        assert c.stats().batched_queries == before

    def test_batched_1024_queries(self, t1):
        """k = 1000 keeps 1250 candidates per query: the main pass runs in 25M-row segments with the buffer cut-back."""
        c = t1.c
        want = t1.ref.topk(t1.q1024, 1000)
        for k in (100, 1000):
            before = c.stats().batched_queries
            res = c.search(t1.q1024, k)
            assert c.stats().batched_queries == before + 1024, f"k={k}: the tensor-core path did not run"
            for qi in range(1024):
                same(res[qi], cut(want[qi], 0, k), f"batched k={k} q{qi}")
            for qi, row in enumerate(T1_PROBES):
                self_match(res[qi], t1, row, f"batched k={k}")

    def test_filters(self, t1):
        c, k = t1.c, 100
        rng = np.random.default_rng(5)
        inc = np.unique(np.concatenate([sample(rng, 1, T1_N + 1, T1_N // 100), np.array(T1_PROBES) + 1]))
        exc = np.unique(np.concatenate([w[0][:1000] for w in self.deep(t1)]))
        for name, kw in (("INCLUDE 1 %", dict(within=inc)), ("EXCLUDE best 1000", dict(excluding=exc))):
            want = t1.ref.topk(t1.q16, k, include=kw.get("within"), exclude=kw.get("excluding"))
            for qi in range(16):
                same(c.search(t1.q16[qi], k, **kw)[0], want[qi], f"{name} single q{qi}")
            before = c.stats().batched_queries
            res = c.search(t1.q16, k, **kw)
            assert c.stats().batched_queries == before + 16, f"{name}: the tensor-core path did not run"
            for qi in range(16):
                same(res[qi], want[qi], f"{name} batched q{qi}")

    def test_pages_past_max_k(self, t1):
        c, k, want = t1.c, 1000, self.deep(t1)
        for qi in range(0, 16, 3):
            cur = None
            for p in range(3):
                res = c.search(t1.q16[qi], k, after=[cur])[0]
                same(res, cut(want[qi], p * k, (p + 1) * k), f"single page {p} q{qi}")
                cur = (res.dist[-1], res.ids[-1])
        curs = [None] * 16
        for p in range(3):
            before = c.stats().batched_queries
            res = c.search(t1.q16, k, after=curs)
            assert c.stats().batched_queries == before + 16, f"page {p}: the tensor-core path did not run"
            for qi in range(16):
                same(res[qi], cut(want[qi], p * k, (p + 1) * k), f"batched page {p} q{qi}")
            curs = [(r.dist[-1], r.ids[-1]) for r in res]

    def test_forced_exact_passes(self, t1):
        c, k, want = t1.c, 100, self.deep(t1)
        c.set_candidate_slack(1)
        try:
            before = c.stats().exact_passes
            for qi in (0, 3, 8, 15):
                same(c.search(t1.q16[qi], k)[0], cut(want[qi], 0, k), f"exact pass q{qi}")
            assert c.stats().exact_passes == before + 4
        finally:
            c.set_candidate_slack(0)

    def test_after_remove_and_replace(self, t1):
        """Remove 1M scattered ids, the tail among them: the holes below n' take the survivors at or above n', in row order
        (DESIGN.md §2).  Then replace 1000 ids, 16 of them with rows close to the queries, and search again."""
        c, ref = t1.c, t1.ref
        rng = np.random.default_rng(17)
        gone = np.unique(np.concatenate([sample(rng, 1, T1_N - 9, 1_000_000 - 10), np.arange(T1_N - 9, T1_N + 1)]))
        gone = gone[~np.isin(gone, np.array(T1_PROBES[:2]) + 1)]
        assert c.remove(gone) == gone.size
        ref.remove(gone)
        n2 = T1_N - gone.size
        assert len(c) == n2
        rows_gone = gone - 1
        holes = rows_gone[rows_gone < n2]
        sources = np.setdiff1d(np.arange(n2, T1_N), rows_gone)
        assert holes.size == sources.size
        for j in np.unique(np.concatenate([rng.integers(0, holes.size, 200), [0, holes.size - 1]])):
            got_id, got_row = c.read_rows(int(holes[j]), 1)
            assert got_id[0] == sources[j] + 1, f"hole {holes[j]} holds id {got_id[0]}, the layout says {sources[j] + 1}"
            assert np.array_equal(got_row[0], ref.row_bytes([sources[j] + 1])[0])

        live = rng.permutation(np.setdiff1d(sample(rng, 1, T1_N + 1, 3000), gone))[:1000]
        new_rows = rng.integers(0, 256, size=(live.size, T1_DIM), dtype=np.uint8)
        new_rows[:16] = np.clip(t1.q16.astype(int) + rng.integers(-3, 4, size=(16, T1_DIM)), 0, 255)
        assert c.replace(live, new_rows) == live.size
        ref.set_rows(live, new_rows)

        want = ref.topk(t1.q16, 2048)
        for k in (100, 2048):
            for qi in range(16):
                same(c.search(t1.q16[qi], k)[0], cut(want[qi], 0, k), f"after removal single k={k} q{qi}")
        k = 1000
        res = c.search(t1.q16, k, after=[(w[1][k - 1], w[0][k - 1]) for w in want])
        for qi in range(16):
            same(res[qi], cut(want[qi], k, 2 * k), f"after removal batched page 2 q{qi}")
        want = ref.topk(t1.q1024, 100)
        before = c.stats().batched_queries
        res = c.search(t1.q1024, 100)
        assert c.stats().batched_queries == before + 1024
        for qi in range(1024):
            same(res[qi], want[qi], f"after removal batched q{qi}")
        inc = np.unique(np.concatenate([live, sample(rng, 1, n2 + 1, n2 // 100)]))
        want = ref.topk(t1.q16, 100, include=inc)
        res = c.search(t1.q16, 100, within=inc)
        for qi in range(16):
            same(res[qi], want[qi], f"after removal INCLUDE q{qi}")


# ---------------------------------------------------------------------------------------------------------------------
# Tier 2: dim 32 over 2^31 + 2^20 rows, across 2^31 and the batched hand-over
# ---------------------------------------------------------------------------------------------------------------------
T2_N, T2_DIM, T2_SEED = 2**31 + 2**20, 32, 31
T2_PROBES = [2**31 - 1, 2**31, 2**31 + 1, T2_N - 1]


@pytest.fixture(scope="class")
def t2():
    t = open_tier(T2_N, T2_DIM, T2_SEED)
    q = synth.synth_queries(77, 64, T2_DIM, T2_N, T2_SEED)
    for i, r in enumerate(T2_PROBES):
        q[i] = synth.synth_rows(T2_SEED, r, 1, T2_DIM)[0]
    t.q64 = q
    t.q8 = np.ascontiguousarray(q[:8])
    yield t
    close_tier(t)


class TestShardAcross2To31:
    def check_64(self, t, batched, what):
        """The 64-query call: through the tensor-core path or query by query, as `batched` says; every answer in full."""
        c = t.c
        want = t.ref.topk(t.q64, 100)
        before = c.stats().batched_queries
        res = c.search(t.q64, 100)
        assert c.stats().batched_queries == before + (64 if batched else 0), \
            f"{what}: {len(c)} rows, the batched path {'should' if batched else 'should not'} run"
        for qi in range(64):
            same(res[qi], want[qi], f"{what} q{qi}")

    def test_searches_across_2_to_31_fall_back(self, t2):
        c = t2.c
        want = cached(t2, "deep8", lambda: t2.ref.topk(t2.q8, 2000))
        for k in (10, 100, 2000):
            for qi in range(8):
                res = c.search(t2.q8[qi], k)[0]
                same(res, cut(want[qi], 0, k), f"single k={k} q{qi}")
                if qi < len(T2_PROBES):
                    self_match(res, t2, T2_PROBES[qi], f"single k={k}")
        self.check_64(t2, False, f"{T2_N} rows")

    def test_filter_page_and_view_above_2_to_31(self, t2):
        c, k = t2.c, 100
        rng = np.random.default_rng(9)
        high = sample(rng, 2**31 + 1, T2_N + 1, 10_000)
        inc = np.unique(np.concatenate([high, np.array(T2_PROBES[1:]) + 1]))
        want = t2.ref.topk(t2.q8, k, include=inc)
        for qi in range(8):
            same(c.search(t2.q8[qi], k, within=inc)[0], want[qi], f"INCLUDE above 2^31 q{qi}")
        deep = cached(t2, "deep8", lambda: t2.ref.topk(t2.q8, 2000))
        for qi in (0, 2, 5):
            cur = None
            for p in range(2):
                res = c.search(t2.q8[qi], 1000, after=[cur])[0]
                same(res, cut(deep[qi], p * 1000, (p + 1) * 1000), f"page {p} q{qi}")
                cur = (res.dist[-1], res.ids[-1])
        vids = np.unique(np.concatenate([high[:999], [T2_PROBES[3] + 1]]))
        want = t2.ref.topk(t2.q8, k, include=vids)
        v = c.view(vids)
        try:
            assert len(v) == 1000
            for qi in range(8):
                same(v.search(t2.q8[qi], k)[0], want[qi], f"view above 2^31 q{qi}")
        finally:
            v.close()

    def test_replace_above_2_to_31_ties_with_a_low_row(self, t2):
        c, ref = t2.c, t2.ref
        row5 = ref.row_bytes([6])
        assert c.replace([2**31 + 8], row5) == 1
        ref.set_rows([2**31 + 8], row5)
        res = c.search(row5[0], 10)[0]
        assert list(res.ids[:2]) == [6, 2**31 + 8] and bits(res.dist[0]) == bits(res.dist[1])
        same(res, ref.topk(row5, 10)[0], "tie across 2^31")

    def test_remove_down_to_the_batched_limit(self, t2):
        """Removing scattered low and high ids down to kBatchMaxRows + 1 rows moves survivors from above 2^31 into the low
        holes; the shard is still one row too long for the batched path.  One more removal brings it in."""
        c, ref = t2.c, t2.ref
        assert len(c) == T2_N, f"{len(c)} rows: this test starts from the filled shard of {T2_N} rows"
        rng = np.random.default_rng(23)
        m = T2_N - (K_BATCH_MAX_ROWS + 1)
        low = sample(rng, 100, 2**30, m // 2)
        high = sample(rng, 2**31 + 17, T2_N - 15, m - m // 2)
        gone = np.unique(np.concatenate([low, high]))
        assert gone.size == m and not np.isin(gone, np.array(T2_PROBES) + 1).any()
        assert c.remove(gone) == m
        ref.remove(gone)
        n2 = K_BATCH_MAX_ROWS + 1
        assert len(c) == n2
        holes = np.sort(gone - 1)
        holes = holes[holes < n2]
        sources = np.setdiff1d(np.arange(n2, T2_N, dtype=np.int64), gone - 1)
        assert holes.size == sources.size and (sources >= 2**31).sum() > m // 3
        pick = np.unique(np.concatenate([rng.integers(0, holes.size, 300), [0, holes.size - 1],
                                         np.nonzero(sources >= 2**31)[0][[0, -1]],
                                         np.nonzero(sources == 2**31 + 7)[0]]))
        for j in pick:
            got_id, got_row = c.read_rows(int(holes[j]), 1)
            assert got_id[0] == sources[j] + 1, f"hole {holes[j]} holds id {got_id[0]}, the layout says {sources[j] + 1}"
            assert np.array_equal(got_row[0], ref.row_bytes([sources[j] + 1])[0]), f"hole {holes[j]}: bytes"
        self.check_64(t2, False, "kBatchMaxRows + 1 rows")

        assert c.remove([50]) == 1
        ref.remove([50])
        assert len(c) == K_BATCH_MAX_ROWS
        self.check_64(t2, True, "kBatchMaxRows rows")

    def test_append_past_the_batched_limit(self, t2):
        c, ref = t2.c, t2.ref
        assert len(c) == K_BATCH_MAX_ROWS, \
            f"{len(c)} rows: this test continues from test_remove_down_to_the_batched_limit, which leaves kBatchMaxRows rows"
        row = np.clip(t2.q64[1:2].astype(int) + 1, 0, 255).astype(np.uint8)
        c.append([2**40], row)
        ref.set_rows([2**40], row)
        assert len(c) == K_BATCH_MAX_ROWS + 1
        self.check_64(t2, False, "kBatchMaxRows + 1 rows after an append")


# ---------------------------------------------------------------------------------------------------------------------
# Tier 3: dim 8 over PBX_MAX_ROWS rows, ids crossing 2^32
# ---------------------------------------------------------------------------------------------------------------------
T3_DIM, T3_SEED, T3_FIRST = 8, 8, 2**31
T3_PROBES = [0, 2**31 - 1, 2**31, PBX_MAX_ROWS - 1]      # local row 2^31 - 1 has id 2^32: ids cross 2^32 there


@pytest.fixture(scope="class")
def t3():
    t = open_tier(PBX_MAX_ROWS, T3_DIM, T3_SEED, T3_FIRST)
    q = synth.synth_queries(55, 8, T3_DIM, PBX_MAX_ROWS, T3_SEED)
    for i, r in enumerate(T3_PROBES):
        q[i] = synth.synth_rows(T3_SEED, T3_FIRST + r, 1, T3_DIM)[0]
    t.q8 = q
    yield t
    close_tier(t)


class TestShardOfMaxRows:
    def deep(self, t):
        return cached(t, "deep", lambda: t.ref.topk(t.q8, 2500))

    def test_searches(self, t3):
        c, want = t3.c, self.deep(t3)
        assert len(c) == PBX_MAX_ROWS
        for k in (10, 100, 2048):
            for qi in range(8):
                res = c.search(t3.q8[qi], k)[0]
                same(res, cut(want[qi], 0, k), f"k={k} q{qi}")
                if qi < len(T3_PROBES):
                    self_match(res, t3, T3_PROBES[qi], f"k={k}")

    def test_exact_pass_filter_and_page(self, t3):
        c, want = t3.c, self.deep(t3)
        c.set_candidate_slack(1)
        try:
            before = c.stats().exact_passes
            same(c.search(t3.q8[1], 100)[0], cut(want[1], 0, 100), "forced exact pass")
            assert c.stats().exact_passes == before + 1
        finally:
            c.set_candidate_slack(0)
        inc = np.unique(np.concatenate([w[0][::2] for w in want]))
        fw = t3.ref.topk(t3.q8, 100, include=inc)
        for qi in range(8):
            same(c.search(t3.q8[qi], 100, within=inc)[0], fw[qi], f"INCLUDE over the top rows q{qi}")
        for qi in (0, 3, 6):
            cur = None
            for p in range(2):
                res = c.search(t3.q8[qi], 1250, after=[cur])[0]
                same(res, cut(want[qi], p * 1250, (p + 1) * 1250), f"page {p} q{qi}")
                cur = (res.dist[-1], res.ids[-1])

    def test_appends_at_the_row_limit(self, t3):
        """At PBX_MAX_ROWS rows every append is refused with PBX_E_CAPACITY and changes nothing, the coalesced single-row
        append (the indexer's) included: queued rows that can never be uploaded would make every later search fail."""
        import torch
        c, ref, q = t3.c, t3.ref, t3.q8
        want = self.deep(t3)
        rng = np.random.default_rng(3)
        d_ids = torch.tensor([2**41], dtype=torch.int64, device="cuda")
        d_row = torch.from_numpy(q[:1].copy()).cuda()
        attempts = [("append of 1 row", lambda: c.append([2**41], q[:1])),
                    ("append of 100 rows", lambda: c.append(np.arange(2**41, 2**41 + 100), np.repeat(q[:1], 100, axis=0))),
                    ("append_device of 1 row", lambda: c.append_device(d_ids.data_ptr(), d_row.data_ptr(), 1))]
        for what, fn in attempts:
            code = error_code(fn)
            after = (code, len(c), error_code(lambda: c.search(q[2], 10)))
            assert after == (PBX_E_CAPACITY, PBX_MAX_ROWS, None), \
                f"{what} at the limit: (status, rows, next search's status) = {after}"
            same(c.search(q[2], 10)[0], cut(want[2], 0, 10), f"search after the refused {what}")

        gone = np.unique(rng.integers(T3_FIRST + 10, T3_FIRST + PBX_MAX_ROWS - 10, 10))
        assert gone.size == 10 and c.remove(gone) == 10
        ref.remove(gone)
        new_ids = np.arange(2**42, 2**42 + 10, dtype=np.int64)
        new_rows = rng.integers(0, 256, size=(10, T3_DIM), dtype=np.uint8)
        for i in range(10):
            c.append(new_ids[i:i + 1], new_rows[i:i + 1])
        ref.set_rows(new_ids, new_rows)
        assert len(c) == PBX_MAX_ROWS
        code = error_code(lambda: c.append([2**43], q[:1]))
        assert (code, len(c)) == (PBX_E_CAPACITY, PBX_MAX_ROWS), f"the 11th append: (status, rows) = {(code, len(c))}"
        got_ids, got_rows = c.read_rows(PBX_MAX_ROWS - 10, 10)         # rows up to 0xFFFFEFFF
        assert list(got_ids) == list(new_ids) and np.array_equal(got_rows, new_rows)
        want = ref.topk(np.concatenate([new_rows, q]), 100)
        for qi in range(18):
            res = c.search(np.concatenate([new_rows, q])[qi], 100)[0]
            same(res, want[qi], f"after the appends at the limit q{qi}")
            if qi < 10:
                assert new_ids[qi] in res.ids[:5].tolist()
