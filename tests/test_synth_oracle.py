"""The complete reference of synthetic corpora (tests/synth_oracle.py) against the CPU oracle, on the CPU.

tests/test_gpu_scale.py trusts this reference at 100M ... 4.29G rows, where nothing else can check a search in full; here
it must agree with synth.py's generator and with oracle.topk over the whole corpus on every case it is used for."""
import numpy as np
import pytest

from oracle import oracle
from pixelbox_b200 import synth
from tests import synth_oracle


@pytest.mark.parametrize("dim", [8, 13, 32, 256])
@pytest.mark.parametrize("first_row", [0, 2**31 - 5, 2**32 - 5, 2**33, 2**40])
def test_torch_generator_matches_synth(dim, first_row):
    seed = 0xC0FFEE ^ dim
    got = synth_oracle.synth_rows_torch(seed, first_row, 37, dim).numpy()
    assert np.array_equal(got, synth.synth_rows(seed, first_row, 37, dim))
    assert np.array_equal(got, oracle.synth_rows(seed, first_row, 37, dim))


def full_answer(rows, ids, queries, k, allowed):
    return [oracle.topk(rows[allowed], ids[allowed], q, k, 1e3) for q in queries]


def same(got, want, what):
    g_ids, g_dist, g_dot, g_n2 = got
    w_ids, w_dist, w_dot, w_n2 = want
    assert list(g_ids) == list(w_ids), f"{what}: ids differ"
    assert np.array_equal(g_dist.view(np.uint32), w_dist.view(np.uint32)), f"{what}: dist bits differ"
    assert np.array_equal(g_dot, w_dot) and np.array_equal(g_n2, w_n2), f"{what}: integer terms differ"


@pytest.mark.parametrize("dim", [8, 32, 256])
def test_reference_equals_the_oracle_over_the_whole_corpus(dim):
    """Small corpora with every feature the scale tests use: a first_row past 2^32, removed ids, replaced rows (one an exact
    copy of another row: a tie at rank k), appended rows (one duplicating a row), INCLUDE and EXCLUDE filters and a deep
    top-K that pages are sliced from.  Several chunks per corpus, so the running top-K is merged across chunks."""
    n, seed, first_row = 6000, 7 + dim, 2**32 - 2000
    rng = np.random.default_rng(dim)
    ref = synth_oracle.SynthReference(n, seed, dim, first_row, chunk_bytes=8 * (dim + 20) * 1500)
    rows = synth.synth_rows(seed, first_row, n, dim)
    ids = np.arange(first_row + 1, first_row + n + 1, dtype=np.int64)
    queries = np.concatenate([rows[[0, 1999, 2000, n - 1]], synth.synth_queries(5, 8, dim, n, seed)[:4],
                              rng.integers(0, 256, size=(4, dim), dtype=np.uint8)])

    # the untouched corpus, and a deep top-K whose slices are pages
    for k in (1, 10, 100, 700):
        for qi, (got, want) in enumerate(zip(ref.topk(queries, k), full_answer(rows, ids, queries, k, slice(None)))):
            same(got, want, f"k={k} q{qi}")

    # removals, replacements (row 17 takes the bytes of row 3: equal dist, ordered by id) and appends (one a copy of row 5)
    gone = rng.choice(ids, 500, replace=False)
    ref.remove(gone)
    rep_ids = np.array([ids[17], ids[40], ids[41]])
    rep_rows = np.stack([rows[3], rng.integers(0, 256, dim, dtype=np.uint8), queries[-1]])
    ref.set_rows(rep_ids, rep_rows)
    app_ids = np.array([first_row + n + 10, first_row + n + 11, 2**45], dtype=np.int64)
    app_rows = np.stack([rows[5], queries[-2], rng.integers(0, 256, dim, dtype=np.uint8)])
    ref.set_rows(app_ids, app_rows)
    cur_rows = rows.copy()
    cur_rows[[17, 40, 41]] = rep_rows
    cur_rows = np.concatenate([cur_rows, app_rows])
    cur_ids = np.concatenate([ids, app_ids])
    live = ~np.isin(cur_ids, gone)
    q2 = np.concatenate([queries, rows[[3, 5]]])
    for k in (10, 300):
        for qi, (got, want) in enumerate(zip(ref.topk(q2, k), full_answer(cur_rows, cur_ids, q2, k, live))):
            same(got, want, f"after mutations k={k} q{qi}")
    tie = ref.topk(rows[3], 2)[0][0]
    assert list(tie) == [ids[3], ids[17]]

    # filters: an INCLUDE set (with ids that are removed or not in the table) and an EXCLUDE set of the best rows
    inc = np.concatenate([rng.choice(cur_ids, 900, replace=False), [1, 2**50]])
    for qi, (got, want) in enumerate(zip(ref.topk(q2, 50, include=inc),
                                         full_answer(cur_rows, cur_ids, q2, 50, live & np.isin(cur_ids, inc)))):
        same(got, want, f"INCLUDE q{qi}")
    exc = np.unique(np.concatenate([r[0] for r in ref.topk(q2, 40)]))
    for qi, (got, want) in enumerate(zip(ref.topk(q2, 60, exclude=exc),
                                         full_answer(cur_rows, cur_ids, q2, 60, live & ~np.isin(cur_ids, exc)))):
        same(got, want, f"EXCLUDE q{qi}")


def test_reference_with_exact_duplicates_and_ties_at_rank_k():
    """A corpus made of few distinct rows repeated (replaced rows), so that many rows tie bit for bit: the answer must cut
    the tie at rank k by id, as the oracle does."""
    n, dim, seed = 3000, 32, 99
    ref = synth_oracle.SynthReference(n, seed, dim, 0, chunk_bytes=8 * (dim + 4) * 700)
    rows = synth.synth_rows(seed, 0, n, dim)
    ids = np.arange(1, n + 1, dtype=np.int64)
    dup = np.arange(100, 3000, 97)
    ref.set_rows(ids[dup], np.repeat(rows[7:8], dup.size, axis=0))
    rows[dup] = rows[7]
    for k in (5, 20, 31, 200):
        got = ref.topk(rows[[7, 8]], k)
        for qi, want in enumerate(full_answer(rows, ids, rows[[7, 8]], k, slice(None))):
            same(got[qi], want, f"k={k} q{qi}")


def test_reference_inside_a_near_duplicate_cluster():
    """2000 rows scattered closely around the query: their f32 distances order them differently from their exact cosines
    (adjacent rows swap), so the k-th best by cos* is often not the k-th best by dist, and the rows that belong to the
    answer lie below it.  The margin's band must catch them at every rank checked."""
    n, dim, seed = 3000, 32, 5
    rng = np.random.default_rng(3)
    rows = synth.synth_rows(seed, 0, n, dim)
    ids = np.arange(1, n + 1, dtype=np.int64)
    base = rows[0].astype(int)
    at = rng.choice(n, 2000, replace=False)
    rows[at] = np.clip(base + rng.integers(-8, 9, size=(2000, dim)), 0, 255).astype(np.uint8)
    ref = synth_oracle.SynthReference(n, seed, dim, 0, chunk_bytes=8 * (dim + 3) * 800)
    ref.set_rows(ids[at], rows[at])
    for k in range(20, 420, 20):
        same(ref.topk(rows[0], k)[0], oracle.topk(rows, ids, rows[0], k, 1e3), f"k={k}")


def test_reference_refuses_a_band_it_cannot_bound():
    """Every row identical: the band around the k-th best holds the whole corpus, which must fail loudly, not slowly."""
    n, dim = 3000, 8
    ref = synth_oracle.SynthReference(n, 1, dim, 0)
    ref.set_rows(np.arange(1, n + 1), np.full((n, dim), 200, np.uint8))
    with pytest.raises(AssertionError, match="rows within the margin"):
        ref.topk(np.full(dim, 200, np.uint8), 10)


def test_margin_is_the_certificate_margin():
    assert synth_oracle.margin(256) == (4 * 256 + 3232) / 2**24
    assert abs(synth_oracle.margin(256) - 2.5e-4) < 1e-5

