"""Hostile inputs for the search's pruning (DESIGN section 5).  Every answer is exact only because every pruning
threshold -- the prep_seed bin, the scan's per-CTA tau and global kappa bin, the batched seed bound, in-pass histogram
thresholds and 32-row block bound, the tighten kernel -- is a lower bound built from at least `keep` real, live, allowed
rows, and because a query whose candidates were dropped (certificate, overflow flag) goes to the exact pass.  A bug there
returns a plausible top-k with a true neighbour missing.  Random, clustered and tied corpora tighten the thresholds early
and never run the rare branches; the corpora here are built to run them:

1. near-duplicates in adversarial row orders: every kappa falls in one bin of the scan's global histogram, so only the
   per-CTA tau prunes, and the CTA buffers are cut back inside the scan loop and after the final filter;
2. near-duplicate clusters larger than the batched candidate buffers (4096 keys, 16384 for keep > 512): the in-pass
   thresholds are bin edges, a cluster inside one bin cannot be cut, the buffer overflows and the query must take the
   exact pass;
3. rows that would beat every live row for their query, at positions >= n (left behind by a shorter load or a removal)
   or excluded by a filter: none of them may feed a threshold or a candidate;
4. extreme image ids (INT64_MIN ... INT64_MAX) in ties that only the id order decides, on every path and in the merges,
   next to the INT64_MAX / +inf padding of unused hit slots.

Every GPU answer is compared with the CPU oracle bit for bit: ids and their order, dist bits, dot, norm2 and the count.
The pure-numpy generators have self-checks that run without a GPU, so that an edit cannot quietly make a case harmless."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import _native as nat

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
I64_MIN, I64_MAX = int(np.iinfo(np.int64).min), int(np.iinfo(np.int64).max)
EXTREME_IDS = np.array([I64_MIN, I64_MIN + 1, -2**32, -1, 0, 1, 2**31 - 1, 2**31, 2**32, I64_MAX - 1, I64_MAX], np.int64)
SINGLE, DEFAULT = 0xFFFFFFFF, 0          # set_batch_min: loop over the single-query scan / the default dispatch
SCAN_HIST_BINS = 4096                    # the single-query scan's global histogram over kappa in [-1, 1]
BATCH_HIST_BINS = 1024                   # the batched path's per-query histogram over kappa in [-1, 1]
BATCH_CAP, BATCH_CAP_LARGE = 4096, 16384  # batched candidate buffer entries per query (keep <= 512 / keep > 512)


# ---- oracle and comparison --------------------------------------------------------------------------------------------
def bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def threads():
    return oracle.max_threads()


def want_topk(rows, ids, queries, k, md):
    return [oracle.topk(rows, ids, q, k, md, threads=threads()) for q in queries]


def prefix(want, k, md):
    """The oracle answer for (k, md) from an answer for a larger k at a larger max_dist: rows with dist < md form a prefix
    of the (dist, id) order (the filter compares the f32 distance with the f64 max_dist)."""
    o_ids, o_dist, o_dot, o_n2 = want
    c = min(k, int(np.count_nonzero(o_dist.astype(np.float64) < md)))
    return o_ids[:c], o_dist[:c], o_dot[:c], o_n2[:c]


def assert_same(res, want, ctx=""):
    o_ids, o_dist, o_dot, o_n2 = want
    assert len(res.ids) == len(o_ids), f"count {len(res.ids)} != {len(o_ids)} {ctx}"
    assert list(res.ids) == list(o_ids), f"ids differ {ctx}"
    assert np.array_equal(bits(res.dist), bits(o_dist)), f"dist bits differ {ctx}"
    assert np.array_equal(res.dot, o_dot), f"dot differs {ctx}"
    assert np.array_equal(res.norm2, o_n2), f"norm2 differs {ctx}"


def check_paths(c, queries, k, md, wants, ctx, modes=(SINGLE, DEFAULT), **filt):
    """Every query both ways: the single-query loop and whatever the default dispatch picks (the tensor-core batched path
    from 2 queries on where the shape allows).  Returns the batched_queries delta of the default dispatch."""
    batched = 0
    for mode in modes:
        c.set_batch_min(mode)
        before = c.stats().batched_queries
        got = c.search(queries, k, md, **filt)
        if mode == DEFAULT:
            batched = c.stats().batched_queries - before
        else:
            assert c.stats().batched_queries == before
        assert len(got) == len(queries)
        for qi in range(len(queries)):
            assert_same(got[qi], wants[qi], f"{ctx} {'single' if mode == SINGLE else 'default'} k={k} md={md} q={qi}")
    c.set_batch_min(DEFAULT)
    return batched


def batched_eligible_rows(keep):
    """Smallest n the batched path takes for `keep` candidates: its seed pass needs 1.5 keep sampled 32-row blocks
    from complete 256-row tiles."""
    return -(-(keep + keep // 2) // 8) * 256


# ---- generators (pure numpy; self-checked below without a GPU) -----------------------------------------------------------
def near_duplicates(rng, n, d, base, moved=3):
    """n rows, each `base` with `moved` bytes moved by +-1..3 (base bytes in [8, 247]: nothing clips)."""
    rows = np.tile(base.astype(np.uint8), (n, 1))
    pos = rng.integers(0, d, size=(n, moved))
    delta = rng.choice(np.array([-3, -2, -1, 1, 2, 3]), size=(n, moved))
    rows[np.arange(n)[:, None], pos] = (base[pos].astype(np.int16) + delta).astype(np.uint8)
    return rows


def adversarial_order(dist, ids, order, chunk=128):
    """Row permutation by oracle (dist, id) to the query.  'worst': worst first, every row at least as close as all rows
    before it (the most pushes and cut-backs of the CTA buffers); 'best': best first; 'saw': ascending inside each
    128-row chunk (the scan's claim unit), chunks from the worst to the best."""
    asc = np.lexsort((ids, dist))
    if order == "best":
        return asc
    desc = asc[::-1]
    if order == "worst":
        return desc
    assert order == "saw"
    return np.concatenate([desc[i:i + chunk][::-1] for i in range(0, len(desc), chunk)])


def adversarial_corpus(seed, n, d, order):
    """(rows, ids, queries): near-duplicates of one base vector in the given row order, ids a random permutation (row
    order is not id order).  Query 0 is the base, query 1 another near-duplicate; the order is by distance to query 0."""
    rng = np.random.default_rng(seed)
    base = rng.integers(8, 248, d).astype(np.uint8)
    rows = near_duplicates(rng, n, d, base)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 7 - 3 * n
    queries = np.stack([base, near_duplicates(rng, 1, d, base)[0]])
    perm = adversarial_order(oracle.all_distances(rows, queries[0]), ids, order)
    return rows[perm], ids[perm], queries


def exact_cosine(q, rows):
    """cos(q, r) in exact integer terms (c(v) = 2v - 255), evaluated in f64."""
    out = np.empty(len(rows))
    for i, r in enumerate(rows):
        dot, nq, nr = oracle.int_terms(q, r)
        out[i] = dot / np.sqrt(float(nq) * float(nr))
    return out


def cluster_corpus(seed, d, n_other, n_cluster, kind, layout, nq=32):
    """(rows, ids, cluster_mask, queries): a cluster of n_cluster rows inside n_other random rows, contiguous or spread
    over the corpus.  kind 'copies': identical rows; 'near': the base with one byte moved by +-1 (an exact cosine spread
    below one bin of the batched histogram).  Queries: cluster members, perturbed members, outsiders."""
    rng = np.random.default_rng(seed)
    n = n_other + n_cluster
    base = rng.integers(8, 248, d).astype(np.uint8)
    if kind == "copies":
        cl = np.tile(base, (n_cluster, 1))
    else:
        cl = np.tile(base, (n_cluster, 1))
        pos = rng.integers(0, d, n_cluster)
        cl[np.arange(n_cluster), pos] = (base[pos].astype(np.int16) + rng.choice([-1, 1], n_cluster)).astype(np.uint8)
    mask = np.zeros(n, bool)
    if layout == "contiguous":
        s = int(rng.integers(0, n_other))
        mask[s:s + n_cluster] = True
    else:
        mask[rng.choice(n, n_cluster, replace=False)] = True
    rows = np.empty((n, d), np.uint8)
    rows[mask] = cl
    rows[~mask] = rng.integers(0, 256, size=(n_other, d), dtype=np.uint8)
    ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64)
    members = rows[rng.choice(np.flatnonzero(mask), nq // 3, replace=False)]
    perturbed = near_duplicates(rng, nq // 3, d, base)
    outsiders = np.concatenate([rows[rng.choice(np.flatnonzero(~mask), 4, replace=False)],
                                rng.integers(0, 256, size=(nq - 2 * (nq // 3) - 4, d), dtype=np.uint8)])
    return rows, ids, mask, np.concatenate([members, perturbed, outsiders])


def poisoned_corpus(seed, n, d, per):
    """(live_rows, live_ids, hostile_rows, hostile_ids, queries).  The live rows sit around one centre X; the queries are
    a live row, a random vector and the antipode of X (every live row is on its cos <= 1e-6 plateau, dist 999999).  For
    every query there are `per` exact copies of it and `per` of its antipode, with ids below every live id: the copies
    beat every live row, and at max_dist > 999999 the antipodes beat every live plateau row on the id order."""
    rng = np.random.default_rng(seed)
    centre = rng.integers(40, 216, d)
    live = np.clip(centre + rng.integers(-40, 41, size=(n, d)), 0, 255).astype(np.uint8)
    live_ids = rng.permutation(np.arange(1, n + 1)).astype(np.int64) * 5
    queries = np.stack([live[int(rng.integers(0, n))], rng.integers(0, 256, d, dtype=np.uint8), (255 - centre).astype(np.uint8)])
    hostile = np.concatenate([np.repeat(queries, per, axis=0), np.repeat((255 - queries).astype(np.uint8), per, axis=0)])
    hostile_ids = -1 - rng.permutation(len(hostile)).astype(np.int64)
    return live, live_ids, hostile, hostile_ids, queries


def extreme_corpus(seed, n=50_000, d=64, group=700):
    """(rows, ids, group_mask, queries): `group` identical rows V whose ids are EXTREME_IDS plus filler from
    [-2^40, 2^40], spread over the corpus; every other row is V plus noise.  Queries: V, V with one byte moved,
    a random vector, and V's antipode (every row on the plateau: the answer is the id order of the whole corpus)."""
    rng = np.random.default_rng(seed)
    v = rng.integers(60, 196, d).astype(np.uint8)
    rows = np.clip(v.astype(int) + rng.integers(-30, 31, size=(n, d)), 0, 255).astype(np.uint8)
    pos = rng.choice(n, group, replace=False)
    rows[pos] = v
    mask = np.zeros(n, bool)
    mask[pos] = True
    ids = np.unique(rng.integers(-2**40, 2**40, size=n + 1000))
    ids = rng.permutation(ids[~np.isin(ids, EXTREME_IDS)])[:n].astype(np.int64)
    ext_pos = np.sort(pos)[np.linspace(0, group - 1, len(EXTREME_IDS)).astype(int)]      # spread over the row range
    ids[ext_pos] = rng.permutation(EXTREME_IDS)
    v1 = v.copy()
    v1[3] += 1
    queries = np.stack([v, v1, rng.integers(0, 256, d, dtype=np.uint8), (255 - v).astype(np.uint8)])
    return rows, ids, mask, queries


# ---- CPU part: the generators do what the GPU tests rely on ---------------------------------------------------------------
@pytest.mark.parametrize("d", [64, 100, 1280])
def test_adversarial_orders_are_what_they_claim(d):
    n = 3000
    for order in ("worst", "best", "saw"):
        rows, ids, queries = adversarial_corpus(11 + d, n, d, order)
        dist = oracle.all_distances(rows, queries[0]).astype(np.float64)
        if order == "worst":
            assert np.all(np.diff(dist) <= 0), "worst-first corpus is not non-increasing in oracle distance"
        elif order == "best":
            assert np.all(np.diff(dist) >= 0)
        else:
            for s in range(0, n, 128):
                assert np.all(np.diff(dist[s:s + 128]) >= 0)
                if s + 128 < n:
                    assert dist[s:s + 128].min() >= dist[s + 128:s + 256].max()
        assert not np.array_equal(np.argsort(ids), np.arange(n)), "row order must not be id order"
        # every kappa of the corpus lies within two bins of the scan's global histogram, for both queries
        for q in queries:
            kap = exact_cosine(q, rows[::7])
            lo, hi = np.floor((kap + 1) * SCAN_HIST_BINS / 2), np.floor((np.minimum(kap, 1 - 1e-12) + 1) * SCAN_HIST_BINS / 2)
            assert hi.max() - lo.min() <= 1, (d, order, kap.min(), kap.max())


@pytest.mark.parametrize("n_cluster,cap", [(9000, BATCH_CAP), (36000, BATCH_CAP_LARGE)])
def test_clusters_exceed_the_batched_buffers(n_cluster, cap):
    for kind in ("copies", "near"):
        rows, ids, mask, queries = cluster_corpus(5, 64, 60_000, n_cluster, kind, "interleaved")
        assert mask.sum() > cap and mask.sum() // 2 > cap, "the cluster (and half of it, for within=) must overflow a buffer"
        cl = rows[mask]
        kap = exact_cosine(cl[0], cl[:: max(1, len(cl) // 500)])
        assert kap.max() - kap.min() < 2 / BATCH_HIST_BINS, "near-copy cluster spread is not below one batched bin"
        # the member and perturbed queries see the whole cluster inside one batched bin
        for q in queries[:20]:
            k2 = exact_cosine(q, cl[::97])
            assert k2.max() - k2.min() < 2 / BATCH_HIST_BINS


def test_poisoned_rows_beat_every_live_row():
    live, live_ids, hostile, hostile_ids, queries = poisoned_corpus(3, 4000, 64, per=8)
    assert hostile_ids.max() < live_ids.min()
    for qi, q in enumerate(queries):
        ld = oracle.all_distances(live, q)
        hd = oracle.all_distances(hostile, q)
        copies = np.flatnonzero(np.all(hostile == q, axis=1))
        assert len(copies) >= 8
        # (dist, id) of every copy is below (dist, id) of every live row
        assert hd[copies].max() < ld.min() or (hd[copies].max() == ld.min() and hostile_ids[copies].max() < live_ids.min())
        if qi == 2:                                                  # the antipode query: every live row on the plateau
            assert np.all(ld == np.float32(999999.0))
            anti = np.flatnonzero(np.all(hostile == 255 - q, axis=1))
            assert np.all(hd[anti] == np.float32(999999.0)) and hostile_ids[anti].max() < live_ids.min()
    # at max_dist 1e7 the whole top-k of every query is hostile when the hostile rows are live
    rows, ids = np.concatenate([live, hostile]), np.concatenate([live_ids, hostile_ids])
    for q in queries:
        assert np.all(oracle.topk(rows, ids, q, 8, 1e7)[0] < 0)


def test_extreme_ids_sit_in_one_tie():
    rows, ids, mask, queries = extreme_corpus(9, n=5000, group=300)
    assert len(np.unique(ids)) == len(ids) and set(EXTREME_IDS.tolist()) <= set(ids[mask].tolist())
    o_ids = oracle.topk(rows, ids, queries[0], 300, 1e3)[0]
    assert list(o_ids) == sorted(ids[mask].tolist()) and o_ids[0] == I64_MIN and o_ids[-1] == I64_MAX
    assert np.all(oracle.all_distances(rows, queries[3]) == np.float32(999999.0))


# ---- 1. adversarial row order: the per-CTA tau, mid-scan and final cut-backs of the scan buffers ------------------------
# (dim, rows, scan CTAs per SM (0: default)).  Rows on both sides of the prep_seed condition (rows >= 8 * 256 * SMs,
# ~303k on 148 SMs).  Every row of these corpora falls in one bin of the global histogram, so a CTA pushes nearly every
# row it sees: its buffer is cut back inside the scan loop once it has seen more than cap - 1024 rows (3072 for
# k <= 1000), after the final filter once it holds more than keep.
ADVERSARIAL = [(64, 200_000, 0), (64, 620_000, 0), (64, 1_600_000, 0),          # compile-time layout, 3 CTAs / SM
               (256, 100_000, 0), (256, 320_000, 0), (256, 520_000, 1),         # one CTA per SM: ~3500 rows per CTA
               (1280, 40_000, 0), (1280, 120_000, 0),                          # x5 layout, split replay at large k
               (100, 60_000, 0), (100, 310_000, 0), (1000, 100_000, 0)]        # ragged rows: scan_generic_kernel exact pass


@gpu
@pytest.mark.parametrize("d,n,per_sm", ADVERSARIAL)
def test_adversarial_row_order(d, n, per_sm):
    from pixelbox_b200.corpus import Corpus
    rows, ids, queries = adversarial_corpus(100 + d, n, d, "best")
    want = want_topk(rows, ids, queries, 2048, 1e3)
    dist0 = oracle.all_distances(rows, queries[0])
    band = float(np.median(dist0))                   # inside the dense band of distances
    with Corpus(d, capacity_hint=n) as c:
        c.set_scan_ctas_per_sm(per_sm)
        for order in ("worst", "best", "saw"):
            perm = adversarial_order(dist0, ids, order)
            c.load(ids[perm], rows[perm])
            for k in (1, 100, 1000, 2048):
                for md in (1e3, band):
                    check_paths(c, queries, k, md, [prefix(w, k, md) for w in want], f"{order} d={d} n={n}")
            if order == "worst" and d in (64, 1000):
                c.set_candidate_slack(1)
                xp = c.stats().exact_passes
                for k in (1, 100):
                    check_paths(c, queries, k, 1e3, [prefix(w, k, 1e3) for w in want], f"slack=1 {order} d={d} n={n}")
                assert c.stats().exact_passes > xp
                c.set_candidate_slack(0)


# ---- 2. clusters larger than the batched candidate buffers: the overflow flag -> exact pass --------------------------------
CLUSTERS = [(d, 100, 60_000, 9_000, kind, layout) for d in (64, 256) for kind in ("copies", "near")
            for layout in ("contiguous", "interleaved")] + \
           [(64, 1000, 64_000, 36_000, "copies", "interleaved"), (256, 1000, 64_000, 36_000, "near", "contiguous")]


@gpu
@pytest.mark.parametrize("d,k,n_other,n_cluster,kind,layout", CLUSTERS)
def test_cluster_larger_than_batched_buffer(d, k, n_other, n_cluster, kind, layout, monkeypatch):
    from pixelbox_b200.corpus import Corpus
    rows, ids, mask, queries = cluster_corpus(200 + d + k, d, n_other, n_cluster, kind, layout)
    nq = len(queries)
    want = want_topk(rows, ids, queries, k, 1e3)
    with Corpus(d) as c:
        c.load(ids, rows)
        for seg in (None, "37"):                 # whole main pass / main pass in segments with cut-backs in between
            if seg:
                monkeypatch.setenv("PBX_BATCH_SEG_TILES", seg)
            xp = c.stats().exact_passes
            modes = (SINGLE, DEFAULT) if seg is None else (DEFAULT,)
            assert check_paths(c, queries, k, 1e3, want, f"seg={seg} {kind} {layout}", modes=modes) == nq, \
                "the tensor-core path did not run"
            assert c.stats().exact_passes > xp
            monkeypatch.delenv("PBX_BATCH_SEG_TILES", raising=False)
        # within= half the cluster (still more rows than a buffer holds) and half of the other rows
        rng = np.random.default_rng(d + k)
        allowed = np.zeros(len(ids), bool)
        allowed[rng.choice(np.flatnonzero(mask), n_cluster // 2, replace=False)] = True
        allowed[rng.choice(np.flatnonzero(~mask), n_other // 2, replace=False)] = True
        want_f = want_topk(rows[allowed], ids[allowed], queries, k, 1e3)
        xp = c.stats().exact_passes
        within = rng.permutation(ids[allowed])
        assert check_paths(c, queries, k, 1e3, want_f, f"within {kind} {layout}", within=within) == nq
        assert c.stats().exact_passes > xp


# ---- 3. poisoned stale and excluded rows -------------------------------------------------------------------------------------
def stale_case(d, n, how):
    """Search n live rows while rows that beat every live row lie at positions >= n ('load': a longer load, then a
    load of the live prefix; 'remove': the hostile tail removed by id) or live but excluded ('exclude').  Single path,
    batched path, candidate slack 1, max_dist 1e3 and 1e7: never a hostile id, always the oracle over the live rows."""
    from pixelbox_b200.corpus import Corpus
    per = 2 * 256                                     # 2 keep: single path k = 100 (keep 256), batched (128), slack 1 (101)
    live, live_ids, hostile, hostile_ids, queries = poisoned_corpus(n + d, n, d, per)
    k = 100
    wants = {md: want_topk(live, live_ids, queries, k, md) for md in (1e3, 1e7)}
    bad = set(hostile_ids.tolist())
    with Corpus(d) as c:
        filt = {}
        if how == "load":
            c.load(np.concatenate([live_ids, hostile_ids]), np.concatenate([live, hostile]))
            c.load(live_ids, live)
        elif how == "remove":
            c.load(np.concatenate([live_ids, hostile_ids]), np.concatenate([live, hostile]))
            assert c.remove(hostile_ids[::-1]) == len(hostile_ids)
        else:
            rng = np.random.default_rng(n)
            at = np.sort(rng.choice(n + len(hostile), len(hostile), replace=False))
            all_rows = np.empty((n + len(hostile), d), np.uint8)
            all_ids = np.empty(n + len(hostile), np.int64)
            mask = np.zeros(len(all_ids), bool)
            mask[at] = True
            all_rows[mask], all_ids[mask] = hostile, hostile_ids
            all_rows[~mask], all_ids[~mask] = live, live_ids
            c.load(all_ids, all_rows)
            filt = {"excluding": rng.permutation(hostile_ids)}
        assert len(c) == (n + len(hostile) if how == "exclude" else n)
        for slack, keep in ((0, 128), (1, k + 1)):      # (keep of the batched path)
            c.set_candidate_slack(slack)
            batched = 0
            for md in (1e3, 1e7):
                batched += check_paths(c, queries, k, md, wants[md], f"{how} d={d} n={n} slack={slack}", **filt)
                for r in c.search(queries, k, md, **filt):
                    assert not bad.intersection(r.ids.tolist())
            eligible = d % 32 == 0 and len(c) >= batched_eligible_rows(keep)
            assert batched == (2 * len(queries) if eligible else 0), (slack, batched, eligible)
        c.set_candidate_slack(0)
        if how == "load":                          # a later append overwrites the stale rows: they become live and win
            c.append(hostile_ids[:per], hostile[:per])
            assert c.search(queries[0], k, 1e3)[0].ids[0] < 0
    return batched


def stale_sizes(sm_count):
    seed_rows = sm_count * 8 * 256                  # prep_seed samples the shard from this many rows on
    eligible = batched_eligible_rows(128)           # k = 100 on the batched path
    return sorted({1025, eligible - 1, eligible, eligible + 1, 20_481, 33_023, 65_535, seed_rows - 1, seed_rows, seed_rows + 1})


@gpu
@pytest.mark.parametrize("how", ["load", "remove", "exclude"])
@pytest.mark.parametrize("d", [64, 100])
def test_poisoned_rows_are_never_read(d, how):
    sizes = stale_sizes(_sm_count()) if d == 64 else [1025, 6143, 33_023]
    # the sizes hit n % 32 in {1, 31}, n % 256 in {1, 255}, n % 1024 in {1, 1023}
    assert {n % 32 for n in sizes} >= {1, 31} and {n % 256 for n in sizes} >= {1, 255} and {n % 1024 for n in sizes} >= {1, 1023}
    for n in sizes:
        stale_case(d, n, how)


@gpu
def test_poisoned_stale_rows_without_vmm():
    """The load variant on plain cudaMalloc buffers (PBX_NO_VMM=1 is read once per process)."""
    code = ("from tests.test_gpu_hostile import stale_case, batched_eligible_rows\n"
            "for n in (1025, batched_eligible_rows(128) + 1, 33_023):\n"
            "    stale_case(64, n, 'load')\n"
            "print('no-vmm ok')\n")
    env = dict(os.environ, PBX_NO_VMM="1", PYTHONPATH=ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert res.returncode == 0 and "no-vmm ok" in res.stdout, res.stdout + res.stderr


def _sm_count():
    from pixelbox_b200.corpus import Corpus
    with Corpus(32) as c:
        return int(c.stats().sm_count)


# ---- 4. extreme ids in ties, on every path --------------------------------------------------------------------------------
@gpu
def test_extreme_ids_in_ties_on_every_path():
    from pixelbox_b200.corpus import Corpus
    rows, ids, mask, queries = extreme_corpus(21)
    n, d, group = rows.shape[0], rows.shape[1], int(mask.sum())
    ks = (5, 100, group - 1, group, group + 50)
    with Corpus(d) as c:
        c.load(ids, rows)
        for slack in (0, 1):                                  # 1: every query takes the exact pass
            c.set_candidate_slack(slack)
            xp = c.stats().exact_passes
            batched = 0
            for k in ks:
                for md in (1e3, 1e-4):                         # 1e-4: only the identical group passes, count < k
                    batched += check_paths(c, queries[:3], k, md, want_topk(rows, ids, queries[:3], k, md), f"slack={slack}")
            assert batched > 0 and c.stats().exact_passes > xp
            top = c.search(queries[0], group + 50, 1e-4)[0]
            assert len(top.ids) == group and top.ids[0] == I64_MIN and top.ids[-1] == I64_MAX
            # the antipode: every row on the 999999 plateau, ordered by id alone
            for k in (100, 2048):
                check_paths(c, queries[2:], k, 1e7, want_topk(rows, ids, queries[2:], k, 1e7), f"plateau slack={slack}")
        c.set_candidate_slack(0)
        # filters made of the extreme ids only
        inside = np.isin(ids, EXTREME_IDS)
        for k in (5, 11, 100):
            for md in (1e3, 1e7):
                check_paths(c, queries, k, md, want_topk(rows[inside], ids[inside], queries, k, md), "within extremes",
                            within=EXTREME_IDS[::-1].copy())
                check_paths(c, queries, k, md, want_topk(rows[~inside], ids[~inside], queries, k, md), "excluding extremes",
                            excluding=EXTREME_IDS)
        # removal of INT64_MIN and INT64_MAX (the removal's sorted-id search at both ends of the range)
        assert c.remove(np.array([I64_MAX, I64_MIN], np.int64)) == 2
        keep = ~np.isin(ids, [I64_MIN, I64_MAX])
        r_ids, r_rows = c.read_rows(0, n - 2)
        assert sorted(r_ids.tolist()) == sorted(ids[keep].tolist())
        for k in (5, group - 2, group):
            for md in (1e3, 1e-4):
                check_paths(c, queries[:3], k, md, want_topk(r_rows, r_ids, queries[:3], k, md), "after remove")
        check_paths(c, queries[2:], 2048, 1e7, want_topk(r_rows, r_ids, queries[2:], 2048, 1e7), "plateau after remove")


@gpu
def test_extreme_ids_across_shards():
    """Three shards on one GPU, the extreme ids split across them: the device merge sees a real INT64_MAX next to the
    INT64_MAX / +inf padding of a shard's unused slots."""
    from pixelbox_b200.corpus import MultiDeviceCorpus
    rows, ids, mask, queries = extreme_corpus(33)
    group = int(mask.sum())
    have = max(1, nat.lib().pbx_device_count())
    with MultiDeviceCorpus(rows.shape[1], [i % have for i in range(3)]) as mc:
        mc.load(ids, rows)
        sizes = [mc.shard_stats(i).rows for i in range(3)]
        bounds = np.cumsum([0] + sizes)
        for lo, hi in zip(bounds[:-1], bounds[1:]):      # (a load splits the rows into contiguous shards)
            assert np.isin(EXTREME_IDS, ids[lo:hi]).any()
        for k, md in ((5, 1e3), (group - 1, 1e3), (group, 1e-4), (2048, 1e-4), (group + 50, 1e3)):
            got = mc.search(queries[:3], k, md)
            for qi, w in enumerate(want_topk(rows, ids, queries[:3], k, md)):
                assert_same(got[qi], w, f"sharded k={k} md={md} q={qi}")
        got = mc.search(queries[3:], 2048, 1e7)
        assert_same(got[0], want_topk(rows, ids, queries[3:], 2048, 1e7)[0], "sharded plateau")
        for filt in ({"within": EXTREME_IDS}, {"excluding": EXTREME_IDS}):
            inside = np.isin(ids, EXTREME_IDS)
            sel = inside if "within" in filt else ~inside
            got = mc.search(queries, 20, 1e7, **filt)
            for qi, w in enumerate(want_topk(rows[sel], ids[sel], queries, 20, 1e7)):
                assert_same(got[qi], w, f"sharded {list(filt)[0]} q={qi}")


@gpu
def test_merges_with_extreme_ids():
    """pbx_merge_hits and pbx_merge_hits_device on lists whose real entries carry INT64_MIN ... INT64_MAX in dist ties,
    short lists padded with (INT64_MAX, +inf): against a plain (dist, signed id) sort of the real entries."""
    import torch
    from pixelbox_b200.corpus import merge_hits
    rng = np.random.default_rng(12)
    n_shards, nq, k = 3, 4, 16
    others = np.setdiff1d(np.unique(rng.integers(-2**40, 2**40, 200)), EXTREME_IDS)
    gathered = np.zeros((n_shards, nq, k), nat.HIT_DTYPE)
    counts = np.zeros((n_shards, nq), np.uint32)
    real = [[] for _ in range(nq)]
    for q in range(nq):
        # the first n_shards * k ids hold every extreme id (query 0 uses them all)
        take = np.concatenate([rng.permutation(np.concatenate([EXTREME_IDS, others[:n_shards * k - len(EXTREME_IDS)]])),
                               rng.permutation(others[n_shards * k - len(EXTREME_IDS):])])
        if q == 1:                                        # query 1: a real INT64_MAX ends shard 0's short list and the merge
            take = np.concatenate([take[take != I64_MAX][:4], [I64_MAX], take[take != I64_MAX][4:]])
        for s in range(n_shards):
            c = ((5, 3, 0)[s] if q == 1 else (k, k - 1, 3, 0)[(s + q) % 4] if q else k)
            sid = take[s * k:s * k + c]
            dist = rng.choice(np.array([0.0, 0.25, 999999.0], np.float32), size=c)
            dist[sid == I64_MAX] = 999999.0
            order = np.lexsort((sid, dist))
            h = gathered[s, q]
            h["image_id"][:c], h["dist"][:c] = sid[order], dist[order]
            h["dot"][:c] = rng.integers(-1000, 1000, c)
            h["norm2"][:c] = s
            h["image_id"][c:], h["dist"][c:] = I64_MAX, np.inf
            counts[s, q] = c
            real[q].extend(h[:c].tolist())
    want_cnt = np.array([min(k, len(r)) for r in real], np.uint32)
    got_hits, got_cnt = merge_hits(gathered, counts, k)
    assert np.array_equal(got_cnt, want_cnt)
    for q in range(nq):
        ref = sorted(real[q], key=lambda h: (h[1], h[0]))[:k]          # (dist, signed id)
        c = int(want_cnt[q])
        assert list(got_hits[q]["image_id"][:c]) == [h[0] for h in ref], q
        assert np.array_equal(bits(got_hits[q]["dist"][:c]), bits([h[1] for h in ref]))
        assert list(got_hits[q]["dot"][:c]) == [h[2] for h in ref]
    assert set(EXTREME_IDS.tolist()) <= {h[0] for h in real[0]}
    assert want_cnt[1] == 8 and got_hits[1]["image_id"][7] == I64_MAX and got_hits[1]["dist"][7] == np.float32(999999.0)
    d_g = torch.from_numpy(gathered.view(np.uint8).reshape(-1)).cuda()
    d_c = torch.from_numpy(counts.astype(np.int32).reshape(-1)).cuda()
    for with_counts in (True, False):
        d_out = torch.zeros(nq * k * 24, dtype=torch.uint8, device="cuda")
        d_cnt = torch.zeros(nq, dtype=torch.int32, device="cuda")
        nat.check(nat.lib().pbx_merge_hits_device(0, d_g.data_ptr(), d_c.data_ptr() if with_counts else None, n_shards, nq, k,
                                                  d_out.data_ptr(), d_cnt.data_ptr(), torch.cuda.current_stream().cuda_stream or 1))
        torch.cuda.synchronize()
        dev = d_out.cpu().numpy().view(nat.HIT_DTYPE).reshape(nq, k)
        assert np.array_equal(d_cnt.cpu().numpy().astype(np.uint32), want_cnt), with_counts
        for q in range(nq):
            c = int(want_cnt[q])
            for f in ("image_id", "dot", "norm2"):
                assert np.array_equal(dev[q][f][:c], got_hits[q][f][:c]), (f, q, with_counts)
            assert np.array_equal(bits(dev[q]["dist"][:c]), bits(got_hits[q]["dist"][:c]))
