"""The search under concurrency.  Every other parity test makes one call at a time, on one stream, from one thread, and
waits before the next; the exactness of the library also rests on ordering machinery those tests never load:

1. the first kernel of a search (prep_seed_kernel, launched with programmatic stream serialisation) reads the caller's
   queries; here a kernel writes them into the same buffer right before every call;
2. searches on different streams share one set of corpus scratch and are chained by an event: here calls of every form
   are enqueued over five streams behind a held stream, with a host-form search in the middle;
3. exact passes tail-launched by the batched finalize: full 1024-query batches in which every query takes one, back to
   back;
4. calls of more than 1024 queries, split into 1024-query chunks (device forms: filter and cursors offset per chunk, a
   last chunk of one query; host forms: a last chunk of one query on the polled single-query path);
5. several threads searching one corpus, every call form at once;
6. removal and growth of the shard with searches in flight;
7. two corpora on one GPU from two threads, and the sharded handle from two threads with a removal in between.

Every answer is compared with the CPU oracle (tests/page_oracle.py for pages and filters) bit for bit: ids in order,
dist bits, dot, norm2 and the count.  Every test also asserts that it ran what it claims: batched_queries and
exact_passes deltas, and streams that were still busy when the later calls were enqueued (a held stream: timing comes
from torch.cuda._sleep, not from chance).  Each case runs once."""
import os
import subprocess
import sys
import threading

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat
from pixelbox_b200.corpus import SearchResult
from tests import page_oracle
from tests.test_gpu_hostile import assert_same, batched_eligible_rows

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
HIT = nat.HIT_DTYPE.itemsize
# count markers of the device forms (include/pixelbox_b200.h): never a valid count
PBX_COUNT_EXCHANGE_TIMEOUT = 0xFFFFFFFF
PBX_COUNT_EXACT_LAUNCH_FAILED = 0xFFFFFFFE
MARKERS = {PBX_COUNT_EXCHANGE_TIMEOUT, PBX_COUNT_EXACT_LAUNCH_FAILED, nat.PBX_COUNT_FILTER_UNSORTED}
HOLD_CYCLES = 100_000_000               # torch.cuda._sleep: ~50 ms at B200 clocks
SEED_ROWS_PER_SM = 8 * 256              # prep_seed samples the shard from rows >= 8 * 256 * SMs on
K, MD = 100, 1e3
SINGLE_KEEP, BATCH_KEEP = 256, 128      # candidates per query at k = 100: single-query scan / batched path
TIE_COPIES, TIE_CURSOR_AT = 400, 10     # paged calls on a tie start after the 10th row of its first page
CHUNK_PROBES = (0, 1023, 1024, 1025, 2047, 2048)


# ---- oracle, device buffers ---------------------------------------------------------------------------------------------
class Oracle:
    """Oracle answers of one table state, computed once per (query bytes, k, max_dist, filter, cursor)."""

    def __init__(self, rows, ids, masks=None):
        self.rows, self.ids, self.masks = rows, ids, masks or {}
        self.cache = {}

    def __call__(self, q, k=K, md=MD, filt=None, after=None):
        key = (np.asarray(q, np.uint8).tobytes(), k, md, filt, None if after is None else (float(after[0]), int(after[1])))
        if key not in self.cache:
            if filt is None and after is None:
                self.cache[key] = oracle.topk(self.rows, self.ids, q, k, md, threads=oracle.max_threads())
            else:
                self.cache[key] = page_oracle.page(self.rows, self.ids, q, k, md, cursor=after,
                                                   allowed=None if filt is None else self.masks[filt])
        return self.cache[key]


class DevOut:
    """[nq][k] pbx_hit records and [nq] counts in device memory."""

    def __init__(self, nq, k=K):
        import torch
        self.nq, self.k = nq, k
        self.hits = torch.zeros(nq * k * HIT, dtype=torch.uint8, device="cuda")
        self.cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")

    def ptrs(self, q0=0):
        return self.hits.data_ptr() + q0 * self.k * HIT, self.cnt.data_ptr() + 4 * q0

    def results(self):
        """After a synchronisation: one SearchResult per query; no count may be a marker."""
        h = self.hits.cpu().numpy().view(nat.HIT_DTYPE).reshape(self.nq, self.k)
        cnt = self.cnt.cpu().numpy().view(np.uint32)
        assert not MARKERS.intersection(cnt.tolist()), f"count markers {sorted(MARKERS.intersection(cnt.tolist()))}"
        assert int(cnt.max()) <= self.k
        return [SearchResult(h[i]["image_id"][:c].copy(), h[i]["dist"][:c].copy(), h[i]["dot"][:c].copy(), h[i]["norm2"][:c].copy())
                for i, c in enumerate(cnt.tolist())]


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def cursors_dev(cur):
    """[nq] HIT_DTYPE cursors -> device memory."""
    return to_dev(np.ascontiguousarray(cur).view(np.uint8))


def cursor_array(after):
    """[(dist, id) or None] -> HIT_DTYPE cursors (None: the first page)."""
    return nat.page_cursors(after, len(after))


def hold(stream):
    """Keeps `stream` busy for ~50 ms: everything enqueued behind it (and behind the search chain) waits."""
    import torch
    with torch.cuda.stream(stream):
        torch.cuda._sleep(HOLD_CYCLES)


def run_threads(fns):
    """Runs every fn in its own thread, released together; re-raises the first failure."""
    errors = []
    gate = threading.Barrier(len(fns))

    def wrap(fn):
        try:
            gate.wait()
            fn()
        except BaseException as e:              # pragma: no cover - reported below
            errors.append(e)

    ts = [threading.Thread(target=wrap, args=(fn,)) for fn in fns]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    if errors:
        raise errors[0]


def probes(nq):
    """Queries checked of an nq-query call: both sides of every 1024-query chunk edge, the last one, every 37th."""
    return sorted({q for q in CHUNK_PROBES if q < nq} | {nq - 1} | set(range(0, nq, 37)))


def sm_count():
    from pixelbox_b200.corpus import Corpus
    with Corpus(32) as c:
        return int(c.stats().sm_count)


# ---- corpora (pure numpy; self-checked below without a GPU) ---------------------------------------------------------------
def random_corpus(seed, n, d=64):
    """(rows, ids): random rows, ids a shuffled range with negative ids among them (row order is not id order)."""
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 3 - n
    return rows, ids


def perturbed(rng, rows, moved=3):
    """Each row with `moved` bytes set to random values: a query whose nearest rows are near its source."""
    out = rows.copy()
    pos = rng.integers(0, rows.shape[1], size=(len(rows), moved))
    out[np.arange(len(rows))[:, None], pos] = rng.integers(0, 256, size=pos.shape, dtype=np.uint8)
    return out


def tie_corpus(seed, n_vec=32, copies=TIE_COPIES, n_other=20_000, d=64):
    """(rows, ids, vecs, others): n_vec random vectors planted `copies` times each, shuffled among n_other random rows.
    A query equal to a planted vector has its whole top-k inside a tie of `copies` rows, more than either path keeps
    (SINGLE_KEEP, 2 * BATCH_KEEP): its certificate fails and it takes the exact pass.  others: random rows (their top-k
    may reach a planted tie too)."""
    rng = np.random.default_rng(seed)
    vecs = rng.integers(0, 256, size=(n_vec, d), dtype=np.uint8)
    other = rng.integers(0, 256, size=(n_other, d), dtype=np.uint8)
    rows = np.concatenate([np.repeat(vecs, copies, axis=0), other])
    perm = rng.permutation(len(rows))
    rows = rows[perm]
    ids = rng.permutation(np.arange(1, len(rows) + 1)).astype(np.int64) * 5 - 7 * len(rows)
    return rows, ids, vecs, other[:64]


def tie_filters(rows, ids, vecs):
    """Filters that keep every planted copy: 'in' = the copies and every other row with an even index; 'ex' = 500 other
    rows.  Returns ({name: sorted ids}, {name: allowed row mask})."""
    planted = (rows[:, None, :] == vecs[None, :, :]).all(axis=2).any(axis=1)
    inc = planted | (np.arange(len(rows)) % 2 == 0)
    exc_ids = ids[~planted][::37][:500]
    masks = {"in": inc, "ex": ~np.isin(ids, exc_ids)}
    sets = {"in": np.sort(ids[inc]), "ex": np.sort(exc_ids)}
    return sets, masks


def tie_cursor(orc, v, filt=None):
    """The cursor of a tie query's second page: the TIE_CURSOR_AT-th row of its first page."""
    o_ids, o_dist, _, _ = orc(v, K, MD, filt)
    return float(o_dist[TIE_CURSOR_AT - 1]), int(o_ids[TIE_CURSOR_AT - 1])


# ---- CPU part: the corpora do what the GPU tests rely on ----------------------------------------------------------------------
def test_tie_corpus_puts_every_top_k_inside_a_tie_larger_than_keep():
    rows, ids, vecs, others = tie_corpus(7)
    sets, masks = tie_filters(rows, ids, vecs)
    assert len(rows) >= batched_eligible_rows(BATCH_KEEP)
    orc = Oracle(rows, ids, masks)
    for v in vecs:
        dist = oracle.all_distances(rows, v)
        for filt in (None, "in", "ex"):
            o_ids, o_dist, _, _ = orc(v, K, MD, filt)
            allowed = np.ones(len(rows), bool) if filt is None else masks[filt]
            tie = allowed & (dist == o_dist[-1])
            assert len(o_ids) == K and np.all(o_dist == o_dist[0]), "the top-k is not one tie"
            assert tie.sum() == TIE_COPIES and tie.sum() > SINGLE_KEEP and tie.sum() >= 2 * BATCH_KEEP
            # the second page, after TIE_CURSOR_AT rows of the tie, still ends inside a tie larger than keep
            cur = tie_cursor(orc, v, filt)
            page = orc(v, K, MD, filt, cur)
            left = tie & ((dist > cur[0]) | (ids > cur[1]))
            assert len(page[0]) == K and page[1][-1] == o_dist[-1] and left.sum() > SINGLE_KEEP
    # the device filters are sorted, as pbx_search_device_filtered requires
    assert all(np.all(np.diff(s) >= 0) for s in sets.values())


def test_chunk_probes_straddle_every_chunk_edge():
    for nq, last in ((1025, 1), (2049, 1), (2500, 452)):
        assert nq % 1024 == last
        p = probes(nq)
        assert {0, nq - 1} <= set(p) and all(e in p for e in range(1024, nq, 1024)) and all(e - 1 in p for e in range(1024, nq, 1024))


# ---- 1. queries written by a kernel right before the call -----------------------------------------------------------------
@gpu
@pytest.mark.parametrize("case", ["single-small", "single-seeded", "batched"])
def test_queries_written_by_a_kernel_just_before_the_call(case):
    """64 rounds on one stream, no synchronisation: index_select (a kernel, not the copy engine) writes query i into
    the same device buffer, then a search reads it.  The search's first kernel computes the query's sum and norm in its
    prologue: if it read query i - 1, the dist bits of query i break."""
    import torch
    from pixelbox_b200.corpus import Corpus
    sms = sm_count()
    seed_rows = SEED_ROWS_PER_SM * sms
    n = 100_000 if case == "single-small" else seed_rows + 17_000
    assert (n >= seed_rows) == (case != "single-small")
    per = 8 if case == "batched" else 1
    rounds, d, k = 64, 64, 50
    rows, ids = random_corpus(11 + len(case), n, d)
    rng = np.random.default_rng(5)
    queries = perturbed(rng, rows[rng.choice(n, rounds * per, replace=False)])
    # every query differs from the one written before it into the same slot in (sum, norm2) of its centred bytes
    cq = queries.astype(np.int64) * 2 - 255
    terms = np.stack([cq.sum(axis=1), (cq * cq).sum(axis=1)], axis=1)
    assert np.all(np.any(terms[per:] != terms[:-per], axis=1))
    orc = Oracle(rows, ids)
    with Corpus(d) as c:
        c.load(ids, rows)
        src = to_dev(queries)
        dq = torch.empty((per, d), dtype=torch.uint8, device="cuda")
        idx = [torch.arange(i * per, (i + 1) * per, device="cuda") for i in range(rounds)]
        out = DevOut(rounds * per, k)
        s = torch.cuda.Stream()
        torch.cuda.synchronize()
        # warm-up: scratch of this shape exists before the loop (its growth would synchronise the device)
        c.search_device(src.data_ptr(), per, k, MD, *out.ptrs(0), s.cuda_stream)
        torch.cuda.synchronize()
        b0 = c.stats().batched_queries
        hold(s)
        with torch.cuda.stream(s):
            for i in range(rounds):
                torch.index_select(src, 0, idx[i], out=dq)
                c.search_device(dq.data_ptr(), per, k, MD, *out.ptrs(i * per), s.cuda_stream)
        assert not s.query(), "the rounds were not enqueued ahead of the device"
        torch.cuda.synchronize()
        assert c.stats().batched_queries - b0 == (rounds * per if per > 1 else 0)
        got = out.results()
        for i, q in enumerate(queries):
            assert_same(got[i], orc(q, k), f"{case} round {i // per} query {i}")


# ---- 2. several streams ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tie_setup():
    rows, ids, vecs, others = tie_corpus(7)
    sets, masks = tie_filters(rows, ids, vecs)
    return rows, ids, vecs, others, sets, Oracle(rows, ids, masks)


def enqueue(c, call, stream):
    """One device-form call: (kind, queries on device, nq, out, extra) with kind single / batched / in / ex / page."""
    kind, dq, nq, out, extra = call
    if kind in ("in", "ex"):
        fids = extra
        c.search_device_filtered(dq.data_ptr(), nq, K, MD, *out.ptrs(), fids.data_ptr(), fids.numel(),
                                 nat.PBX_FILTER_INCLUDE if kind == "in" else nat.PBX_FILTER_EXCLUDE, stream=stream)
    elif kind == "page":
        c.search_device_page(dq.data_ptr(), nq, K, MD, *out.ptrs(), extra[0].data_ptr(), stream=stream)
    else:
        c.search_device(dq.data_ptr(), nq, K, MD, *out.ptrs(), stream=stream)


def want_of(orc, call, queries):
    kind, _, _, _, extra = call
    if kind in ("in", "ex"):
        return [orc(q, K, MD, kind) for q in queries]
    if kind == "page":
        return [orc(q, K, MD, None, a) for q, a in zip(queries, extra[1])]
    return [orc(q, K, MD) for q in queries]


@gpu
def test_calls_on_several_streams_behind_a_held_stream(tie_setup):
    """Every device form enqueued over streams A, B, C, the corpus' own stream and the legacy stream while A is held:
    every call waits for its predecessor through the chained event.  A host-form search (single and batched) in the
    middle waits for the device calls and does not disturb them."""
    import torch
    from pixelbox_b200.corpus import Corpus
    rows, ids, vecs, others, sets, orc = tie_setup
    A, B, C = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    streams = [A.cuda_stream, B.cuda_stream, C.cuda_stream, None, 0]
    tq = np.concatenate([vecs[:8], others[:8]])          # 8 tie queries (exact pass), 8 random ones
    d_tq = to_dev(tq)
    after = [tie_cursor(orc, v) for v in vecs[:8]] + [None] * 8
    d_in, d_ex = to_dev(sets["in"]), to_dev(sets["ex"])

    def plan():
        # (kind, device queries, nq, out, extra), the host queries, the number of tie queries in it
        def q(i, j):
            return d_tq[i:j], tq[i:j]
        calls = []
        for kind, (i, j) in (("single", (0, 1)), ("batched", (0, 16)), ("in", (4, 12)), ("ex", (1, 2)), ("page", (0, 16)),
                             ("single", (8, 9)), ("page", (2, 3)), ("batched", (3, 13)), ("ex", (0, 16)), ("single", (3, 4))):
            dq, hq = q(i, j)
            extra = {"in": d_in, "ex": d_ex}.get(kind)
            if kind == "page":
                extra = (cursors_dev(cursor_array(after[i:j])), after[i:j])
            calls.append(((kind, dq, j - i, DevOut(j - i), extra), hq, sum(1 for x in range(i, j) if x < 8)))
        return calls

    with Corpus(rows.shape[1]) as c:
        c.load(ids, rows)
        warm, first, second = plan(), plan(), plan()
        torch.cuda.synchronize()                          # (torch fills and copies run on the legacy stream)
        for call, _, _ in warm:                           # warm-up: every scratch buffer at its size
            enqueue(c, call, A.cuda_stream)
        c.search(tq[:1], K)
        c.search(tq, K)
        torch.cuda.synchronize()
        st0 = c.stats()
        hold(A)
        for j, (call, _, _) in enumerate(first):
            enqueue(c, call, streams[j % len(streams)])
        assert not A.query(), "the calls were not enqueued behind the held stream"
        host_single = c.search(tq[0], K)[0]               # waits for every call before it
        host_batch = c.search(tq, K)
        hold(A)
        for j, (call, _, _) in enumerate(second):
            enqueue(c, call, streams[(j + 2) % len(streams)])
        assert not A.query()
        torch.cuda.synchronize()
        st1 = c.stats()
        n_batched = sum(call[2] for call, _, _ in first + second if call[2] > 1) + len(tq)
        assert st1.batched_queries - st0.batched_queries == n_batched
        n_tie = sum(t for _, _, t in first + second) + 1 + 8
        assert st1.exact_passes - st0.exact_passes >= n_tie, (st1.exact_passes - st0.exact_passes, n_tie)
        for half, calls in (("before", first), ("after", second)):
            for j, (call, hq, _) in enumerate(calls):
                for qi, (g, w) in enumerate(zip(call[3].results(), want_of(orc, call, hq))):
                    assert_same(g, w, f"{half} the host search: call {j} ({call[0]}) query {qi}")
        assert_same(host_single, orc(tq[0]), "host single")
        for qi, q in enumerate(tq):
            assert_same(host_batch[qi], orc(q), f"host batch query {qi}")


# ---- 3. back-to-back exact passes at full batch size ------------------------------------------------------------------------
@gpu
def test_back_to_back_exact_passes_at_full_batch(tie_setup):
    """Three 1024-query batched calls in which every query takes the exact pass (tail-launched by the finalize kernel),
    then batched -> single -> batched filtered -> single paged, on one stream without synchronisation."""
    import torch
    from pixelbox_b200.corpus import Corpus
    rows, ids, vecs, others, sets, orc = tie_setup
    rng = np.random.default_rng(3)
    nq = 1024
    pick = rng.integers(0, len(vecs), size=(5, nq))
    batches = [vecs[p] for p in pick]
    d_batches = [to_dev(b) for b in batches]
    d_in = to_dev(sets["in"])
    v_single, v_page = vecs[int(pick[0, 7])], vecs[int(pick[1, 9])]
    cur = tie_cursor(orc, v_page)
    d_single, d_page = to_dev(v_single[None]), to_dev(v_page[None])
    d_cur = cursors_dev(cursor_array([cur]))
    s = torch.cuda.Stream()
    outs = [DevOut(nq) for _ in range(4)] + [DevOut(1), DevOut(nq), DevOut(1)]

    def run():
        for i in range(3):
            c.search_device(d_batches[i].data_ptr(), nq, K, MD, *outs[i].ptrs(), s.cuda_stream)
        c.search_device(d_batches[3].data_ptr(), nq, K, MD, *outs[3].ptrs(), s.cuda_stream)
        c.search_device(d_single.data_ptr(), 1, K, MD, *outs[4].ptrs(), s.cuda_stream)
        c.search_device_filtered(d_batches[4].data_ptr(), nq, K, MD, *outs[5].ptrs(), d_in.data_ptr(), d_in.numel(),
                                 nat.PBX_FILTER_INCLUDE, stream=s.cuda_stream)
        c.search_device_page(d_page.data_ptr(), 1, K, MD, *outs[6].ptrs(), d_cur.data_ptr(), stream=s.cuda_stream)

    with Corpus(rows.shape[1]) as c:
        c.load(ids, rows)
        torch.cuda.synchronize()
        run()                                            # warm-up: scratch at its size
        torch.cuda.synchronize()
        st0 = c.stats()
        hold(s)
        run()
        assert not s.query(), "the calls were not enqueued back to back"
        torch.cuda.synchronize()
        st1 = c.stats()
        total = 5 * nq + 2
        assert st1.batched_queries - st0.batched_queries == 5 * nq
        assert st1.exact_passes - st0.exact_passes == total, (st1.exact_passes - st0.exact_passes, total)
        for i in range(4):
            for qi, (g, q) in enumerate(zip(outs[i].results(), batches[i])):
                assert_same(g, orc(q), f"batch {i} query {qi}")
        assert_same(outs[4].results()[0], orc(v_single), "single")
        for qi, (g, q) in enumerate(zip(outs[5].results(), batches[4])):
            assert_same(g, orc(q, K, MD, "in"), f"filtered batch query {qi}")
        assert_same(outs[6].results()[0], orc(v_page, K, MD, None, cur), "single paged")


# ---- 4. calls of more than 1024 queries ----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def wide_setup():
    n, d, k = 60_000, 64, 20
    rows, ids = random_corpus(41, n, d)
    rng = np.random.default_rng(42)
    src = rng.integers(0, n, 2500)
    queries = perturbed(rng, rows[src], moved=2)
    allowed = rng.random(n) < 0.5
    # one cursor per query: its distance to its source row (near the top of its order)
    after = [(float(oracle.cosine_distance(q, rows[r])), int(ids[r])) for q, r in zip(queries, src)]
    return rows, ids, queries, np.sort(ids[allowed]), after, Oracle(rows, ids, {"in": allowed}), k


@gpu
@pytest.mark.parametrize("nq", [1025, 2049, 2500])
def test_device_forms_past_1024_queries(nq, wide_setup):
    """Device forms split into 1024-query chunks: the queries, hits, counts, filter and cursors of every chunk are offset,
    the last chunk (1, 1 and 452 queries) has its own launch plan."""
    import torch
    from pixelbox_b200.corpus import Corpus
    rows, ids, queries, in_ids, after, orc, k = wide_setup
    q = queries[:nq]
    dq, d_in = to_dev(q), to_dev(in_ids)
    d_cur = cursors_dev(cursor_array(after[:nq]))
    with Corpus(rows.shape[1]) as c:
        c.load(ids, rows)
        assert len(c) >= batched_eligible_rows(32)
        outs = {f: DevOut(nq, k) for f in ("plain", "in", "page")}
        torch.cuda.synchronize()
        b0 = c.stats().batched_queries
        c.search_device(dq.data_ptr(), nq, k, MD, *outs["plain"].ptrs())
        c.search_device_filtered(dq.data_ptr(), nq, k, MD, *outs["in"].ptrs(), d_in.data_ptr(), d_in.numel(), nat.PBX_FILTER_INCLUDE)
        c.search_device_page(dq.data_ptr(), nq, k, MD, *outs["page"].ptrs(), d_cur.data_ptr())
        c.synchronize()
        torch.cuda.synchronize()
        assert c.stats().batched_queries - b0 == 3 * nq
        got = {f: o.results() for f, o in outs.items()}
        for i in probes(nq):
            assert_same(got["plain"][i], orc(q[i], k), f"nq={nq} plain query {i}")
            assert_same(got["in"][i], orc(q[i], k, MD, "in"), f"nq={nq} filtered query {i}")
            assert_same(got["page"][i], orc(q[i], k, MD, None, after[i]), f"nq={nq} paged query {i}")


@gpu
def test_host_forms_past_1024_queries(wide_setup):
    """Host forms at 1025 queries: a batched chunk of 1024, then one query on the polled single-query path."""
    from pixelbox_b200.corpus import Corpus
    rows, ids, queries, in_ids, after, orc, k = wide_setup
    nq = 1025
    q = queries[:nq]
    rng = np.random.default_rng(8)
    within = rng.permutation(in_ids)
    with Corpus(rows.shape[1]) as c:
        c.load(ids, rows)
        calls = {
            "search": lambda: c.search(q, k),
            "hits": lambda: _hits_to_results(*c.search_hits(q, k)),
            "within": lambda: c.search(q, k, within=within),
            "after": lambda: c.search(q, k, after=after[:nq]),
        }
        for name, fn in calls.items():
            b0 = c.stats().batched_queries
            got = fn()
            assert c.stats().batched_queries - b0 == 1024, name
            assert len(got) == nq
            for i in probes(nq):
                want = orc(q[i], k, MD, "in" if name == "within" else None, after[i] if name == "after" else None)
                assert_same(got[i], want, f"{name} query {i}")


def _hits_to_results(hits, cnt):
    return [SearchResult(hits[i]["image_id"][:c].copy(), hits[i]["dist"][:c].copy(), hits[i]["dot"][:c].copy(), hits[i]["norm2"][:c].copy())
            for i, c in enumerate(cnt.tolist())]


# ---- 5. threads ---------------------------------------------------------------------------------------------------------------
@gpu
def test_threads_search_one_corpus(tie_setup):
    """Four threads with fixed scripts on one Corpus at once -- one query (polled path), eight (batched), filtered, paged
    and search_hits -- and a fifth making device-form calls on its own stream."""
    import torch
    from pixelbox_b200.corpus import Corpus
    rows, ids, vecs, others, sets, orc = tie_setup
    pool = np.concatenate([vecs[:8], others[:16]])        # 8 tie queries, 16 random ones
    pool_after = [tie_cursor(orc, v) for v in vecs[:8]] + [None] * 16
    for q in pool:                                        # every oracle answer before the threads start
        for filt in (None, "in", "ex"):
            orc(q, K, MD, filt)
    for q, a in zip(pool, pool_after):
        orc(q, K, MD, None, a)
    seen = {t: [] for t in ("single", "batched", "filtered", "paged", "device")}   # (queries, filt, cursors, results)

    def single():
        for r in range(16):
            q = pool[(3 * r) % len(pool)]
            seen["single"].append(([q], None, None, c.search(q, K)))

    def batched():
        for r in range(8):
            sel = [(r + 5 * j) % len(pool) for j in range(8)]
            seen["batched"].append((pool[sel], None, None, c.search(pool[sel], K)))

    def filtered():
        for r in range(8):
            sel = [(2 * r + 7 * j) % len(pool) for j in range(4)]
            filt = "in" if r % 2 == 0 else "ex"
            kw = {"within": sets["in"][::-1]} if filt == "in" else {"excluding": sets["ex"]}
            seen["filtered"].append((pool[sel], filt, None, c.search(pool[sel], K, **kw)))

    def paged():
        for r in range(8):
            sel = [(r + 11 * j) % len(pool) for j in range(3 if r % 2 == 0 else 2)]
            if r % 2 == 0:
                cur = [pool_after[i] for i in sel]
                seen["paged"].append((pool[sel], None, cur, c.search(pool[sel], K, after=cur)))
            else:
                seen["paged"].append((pool[sel], None, None, _hits_to_results(*c.search_hits(pool[sel], K))))

    s = torch.cuda.Stream()
    d_pool, d_ex = to_dev(pool), to_dev(sets["ex"])
    dev_outs = [DevOut(len(pool)) for _ in range(8)]
    torch.cuda.synchronize()

    def device():
        for r, out in enumerate(dev_outs):
            if r % 2 == 0:
                c.search_device(d_pool.data_ptr(), len(pool), K, MD, *out.ptrs(), s.cuda_stream)
            else:
                c.search_device_filtered(d_pool.data_ptr(), len(pool), K, MD, *out.ptrs(), d_ex.data_ptr(), d_ex.numel(),
                                         nat.PBX_FILTER_EXCLUDE, stream=s.cuda_stream)
        s.synchronize()
        for r, out in enumerate(dev_outs):
            seen["device"].append((pool, None if r % 2 == 0 else "ex", None, out.results()))

    with Corpus(rows.shape[1]) as c:
        c.load(ids, rows)
        st0 = c.stats()
        run_threads([single, batched, filtered, paged, device])
        torch.cuda.synchronize()
        st1 = c.stats()
        n_batched = sum(len(qs) for t, calls in seen.items() if t != "single" for qs, _, _, _ in calls)
        assert st1.batched_queries - st0.batched_queries == n_batched
        n_tie = sum(sum(1 for q in qs if any(np.array_equal(q, v) for v in vecs)) for calls in seen.values() for qs, _, _, _ in calls)
        assert n_tie > 100 and st1.exact_passes - st0.exact_passes >= n_tie
        for t, calls in seen.items():
            for j, (qs, filt, cur, res) in enumerate(calls):
                assert len(res) == len(qs)
                for i, q in enumerate(qs):
                    assert_same(res[i], orc(q, K, MD, filt, None if cur is None else cur[i]), f"thread {t} call {j} query {i}")


# ---- 6. removal and growth with searches in flight ------------------------------------------------------------------------------
@gpu
def test_removal_orders_after_calls_on_two_held_streams():
    """Device calls of every form on two held streams, then remove() with no synchronisation, then the same calls again:
    the calls enqueued before the removal see the whole table, the ones after it the table without the removed rows."""
    import torch
    from pixelbox_b200.corpus import Corpus
    n, d, k = 120_000, 64, 50
    rows, ids = random_corpus(61, n, d)
    rng = np.random.default_rng(62)
    src = rng.choice(n, 16, replace=False)
    queries = perturbed(rng, rows[src], moved=2)
    gone = rng.random(n) < 0.2
    gone[src[::2]] = True                                  # half the queries lose their nearest row
    inc = rng.random(n) < 0.5
    inc_ids = np.sort(ids[inc])
    after = [(float(oracle.cosine_distance(q, rows[r])), int(ids[r])) if i % 3 else None for i, (q, r) in enumerate(zip(queries, src))]
    pre = Oracle(rows, ids, {"in": inc})
    post = Oracle(rows[~gone], ids[~gone], {"in": inc[~gone]})
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    dq, d_in, d_cur = to_dev(queries), to_dev(inc_ids), cursors_dev(cursor_array(after))

    shape = (("single", 1), ("batched", 16), ("in", 16), ("page", 16), ("single", 1), ("page", 1))
    out_sets = [[DevOut(nq, k) for _, nq in shape] for _ in range(3)]

    def calls(orc, outs):
        out = []
        for j, ((kind, nq), o) in enumerate(zip(shape, outs)):
            stream = (A if j % 2 == 0 else B).cuda_stream
            if kind == "in":
                c.search_device_filtered(dq.data_ptr(), nq, k, MD, *o.ptrs(), d_in.data_ptr(), d_in.numel(), nat.PBX_FILTER_INCLUDE, stream=stream)
            elif kind == "page":
                c.search_device_page(dq.data_ptr(), nq, k, MD, *o.ptrs(), d_cur.data_ptr(), stream=stream)
            else:
                c.search_device(dq.data_ptr(), nq, k, MD, *o.ptrs(), stream)
            out.append((kind, nq, o, orc))
        return out

    def check(enqueued, when):
        for kind, nq, o, orc in enqueued:
            for i, g in enumerate(o.results()):
                want = orc(queries[i], k, MD, "in" if kind == "in" else None, after[i] if kind == "page" else None)
                assert_same(g, want, f"{when} the removal: {kind} nq={nq} query {i}")

    with Corpus(d) as c:
        c.load(ids, rows)
        torch.cuda.synchronize()
        calls(pre, out_sets[0])                            # warm-up: scratch at its size
        torch.cuda.synchronize()
        b0 = c.stats().batched_queries
        hold(A)
        hold(B)
        before = calls(pre, out_sets[1])
        assert not A.query() and not B.query()
        assert c.remove(ids[gone]) == int(gone.sum())      # no synchronisation before this
        assert A.query() and B.query(), "the removal returned before the searches enqueued ahead of it had finished"
        after_calls = calls(post, out_sets[2])
        torch.cuda.synchronize()
        assert c.stats().batched_queries - b0 == 2 * (16 + 16 + 16)
        check(before, "before")
        check(after_calls, "after")
        assert len(c) == n - int(gone.sum())


@gpu
def test_host_searches_see_all_of_a_removal_or_none():
    """One thread removes a set of ids and re-appends part of them while another makes host searches: every answer is
    the oracle's answer over one of the three table states, never a partly removed table."""
    from pixelbox_b200.corpus import Corpus
    n, d, k = 200_000, 64, 20
    rows, ids = random_corpus(71, n, d)
    rng = np.random.default_rng(72)
    gone = np.zeros(n, bool)
    gone[rng.choice(n, 20_000, replace=False)] = True
    g_idx = np.flatnonzero(gone)
    back = g_idx[: len(g_idx) // 2]
    queries = perturbed(rng, rows[np.concatenate([g_idx[:2], back[-2:], rng.choice(np.flatnonzero(~gone), 2)])], moved=1)
    states = [Oracle(rows, ids), Oracle(rows[~gone], ids[~gone]),
              Oracle(np.concatenate([rows[~gone], rows[back]]), np.concatenate([ids[~gone], ids[back]]))]
    # the three states give different answers: query 0 loses its source row, query 2 gets it back
    assert not _same_want(states[0](queries[0], k), states[1](queries[0], k))
    assert not _same_want(states[1](queries[2], k), states[2](queries[2], k))
    for st in states:
        for q in queries:
            st(q, k)
    seen = []
    started, done = threading.Event(), threading.Event()

    def writer():
        try:
            started.wait(60)                              # the reader has seen the whole table
            assert c.remove(ids[gone]) == len(g_idx)
            c.append(ids[back], rows[back])
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
        c.search(queries[0], k)                           # warm-up of both shapes
        c.search(queries, k)
        run_threads([writer, reader])
        assert len(c) == n - len(g_idx) + len(back)
        hit = set()
        for j, (qis, res) in enumerate(seen):
            match = [st for st in range(3) if all(_same(res[i], states[st](queries[qi], k)) for i, qi in enumerate(qis))]
            assert match, f"search {j} matches no table state"
            hit.update(match)
        assert {0, 2} <= hit, hit                         # searches ran before the removal and after the re-append
        for qi, q in enumerate(queries):
            assert_same(c.search(q, k)[0], states[2](q, k), f"final query {qi}")


def _same(res, want):
    o_ids, o_dist, o_dot, o_n2 = want
    return (len(res.ids) == len(o_ids) and list(res.ids) == list(o_ids) and np.array_equal(res.dist.view(np.uint32), o_dist.view(np.uint32))
            and np.array_equal(res.dot, o_dot) and np.array_equal(res.norm2, o_n2))


def growth_case(mapped):
    """Appends that grow the shard while device searches are pending on a held stream.  Mapped growth leaves the buffers
    in place; the cudaMalloc fallback (PBX_NO_VMM=1) waits for the device, moves the buffers and the batched path must
    rebuild its tensor map.  The in-flight searches see the old rows, a batched search right
    after the growth the new ones."""
    import torch
    from pixelbox_b200.corpus import Corpus
    n0, n1, d, k = 100_000, 40_000, 256, 30
    rows, ids = random_corpus(81, n0 + n1, d)
    rng = np.random.default_rng(82)
    src = np.concatenate([rng.choice(n0, 8, replace=False), n0 + rng.choice(n1, 8, replace=False)])
    queries = perturbed(rng, rows[src], moved=4)
    old, new = Oracle(rows[:n0], ids[:n0]), Oracle(rows, ids)
    for st in (old, new):
        for q in queries:
            st(q, k)
    dq = to_dev(queries)
    s = torch.cuda.Stream()
    with Corpus(d, capacity_hint=16) as c:
        assert c.stats().reserved == (1 if mapped else 0)
        c.load(ids[:n0], rows[:n0])
        cap0 = c.stats().capacity_rows
        assert cap0 < n0 + n1
        outs = [DevOut(1, k), DevOut(16, k), DevOut(16, k)]
        c.search_device(dq.data_ptr(), 16, k, MD, *outs[1].ptrs(), s.cuda_stream)    # warm-up
        torch.cuda.synchronize()
        b0 = c.stats().batched_queries
        hold(s)
        c.search_device(dq.data_ptr(), 1, k, MD, *outs[0].ptrs(), s.cuda_stream)
        c.search_device(dq.data_ptr(), 16, k, MD, *outs[1].ptrs(), s.cuda_stream)
        assert not s.query(), "the growth must begin while the searches are pending"
        c.append(ids[n0:], rows[n0:])
        if not mapped:                                     # the fallback frees the old buffers: it must wait for the searches
            assert s.query(), "the buffers moved under pending searches"
        c.search_device(dq.data_ptr(), 16, k, MD, *outs[2].ptrs(), s.cuda_stream)
        torch.cuda.synchronize()
        st = c.stats()
        assert st.capacity_rows > cap0 and st.rows == n0 + n1
        assert st.batched_queries - b0 == 32
        assert_same(outs[0].results()[0], old(queries[0], k), "in flight, single")
        for i, g in enumerate(outs[1].results()):
            assert_same(g, old(queries[i], k), f"in flight, batched query {i}")
        for i, g in enumerate(outs[2].results()):
            assert_same(g, new(queries[i], k), f"after the growth, batched query {i}")


@gpu
def test_growth_with_searches_in_flight_mapped():
    growth_case(True)


@gpu
def test_growth_with_searches_in_flight_without_vmm():
    code = ("from tests.test_gpu_concurrency import growth_case\n"
            "growth_case(False)\n"
            "print('no-vmm ok')\n")
    env = dict(os.environ, PBX_NO_VMM="1", PYTHONPATH=ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=280)
    assert res.returncode == 0 and "no-vmm ok" in res.stdout, res.stdout + res.stderr


# ---- 7. two corpora on one GPU; the sharded handle ------------------------------------------------------------------------------
@gpu
def test_two_corpora_searched_from_two_threads(tie_setup):
    """One corpus on the batched path with exact passes, another on the single-query path, searched at the same time."""
    from pixelbox_b200.corpus import Corpus
    rows, ids, vecs, others, sets, orc = tie_setup
    rows2, ids2 = random_corpus(91, 80_000, 128)
    rng = np.random.default_rng(92)
    q2 = perturbed(rng, rows2[rng.choice(len(rows2), 24, replace=False)])
    orc2 = Oracle(rows2, ids2)
    batches = [vecs[rng.integers(0, len(vecs), 64)] for _ in range(6)]
    for q in q2:
        orc2(q, 40)
    got1, got2 = [], []
    with Corpus(rows.shape[1]) as c1, Corpus(rows2.shape[1]) as c2:
        c1.load(ids, rows)
        c2.load(ids2, rows2)
        s1, s2 = c1.stats(), c2.stats()
        run_threads([lambda: got1.extend(c1.search(b, K) for b in batches),
                     lambda: got2.extend(c2.search(q, 40)[0] for q in q2)])
        t1, t2 = c1.stats(), c2.stats()
        assert t1.batched_queries - s1.batched_queries == 6 * 64
        assert t1.exact_passes - s1.exact_passes == 6 * 64
        assert t2.batched_queries == s2.batched_queries
        for b, res in zip(batches, got1):
            for i, q in enumerate(b):
                assert_same(res[i], orc(q), f"batched corpus query {i}")
        for i, q in enumerate(q2):
            assert_same(got2[i], orc2(q, 40), f"single-path corpus query {i}")


@gpu
def test_sharded_handle_searched_from_two_threads_with_a_removal():
    """A 3-shard MultiDeviceCorpus on device 0 searched from two threads at once while a third removes rows: every
    answer is the oracle's over the table before or after the removal."""
    from pixelbox_b200.corpus import MultiDeviceCorpus
    n, d, k = 90_000, 64, 25
    rows, ids = random_corpus(101, n, d)
    rng = np.random.default_rng(102)
    gone = rng.random(n) < 0.1
    src = np.concatenate([rng.choice(np.flatnonzero(gone), 3, replace=False), rng.choice(np.flatnonzero(~gone), 3, replace=False)])
    queries = perturbed(rng, rows[src], moved=1)
    states = [Oracle(rows, ids), Oracle(rows[~gone], ids[~gone])]
    for st in states:
        for q in queries:
            st(q, k)
    assert not all(_same_want(states[0](q, k), states[1](q, k)) for q in queries)
    seen = [[], []]
    started = [threading.Event(), threading.Event()]
    removed = threading.Event()

    def searcher(t):
        def run():
            r = 0
            while not removed.is_set() or r < 12:
                sel = [r % len(queries)] if t == 0 else list(range(len(queries)))
                seen[t].append((sel, mc.search(queries[sel], k)))
                r += 1
                if r == 3:
                    started[t].set()
            started[t].set()
        return run

    def remover():
        try:
            for e in started:                             # both searchers are running
                e.wait(60)
            assert mc.remove(ids[gone]) == int(gone.sum())
        finally:
            removed.set()

    with MultiDeviceCorpus(d, [0, 0, 0]) as mc:
        mc.load(ids, rows)
        assert [mc.shard_stats(i).rows > 0 for i in range(3)] == [True] * 3
        run_threads([searcher(0), searcher(1), remover])
        hit = set()
        for t in range(2):
            for j, (sel, res) in enumerate(seen[t]):
                match = [st for st in range(2) if all(_same(res[i], states[st](queries[qi], k)) for i, qi in enumerate(sel))]
                assert match, f"thread {t} search {j} matches neither table state"
                hit.update(match)
        assert hit == {0, 1}
        got = mc.search(queries, k)
        for i, q in enumerate(queries):
            assert_same(got[i], states[1](q, k), f"sharded after the removal, query {i}")


def _same_want(a, b):
    return list(a[0]) == list(b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))
