"""Range oracle of the range searches: the similarity SQL without its LIMIT

    SELECT image_id, cosine_distance(?, hash) AS dist FROM semantic_hashes
    WHERE dist < :max_dist [AND (dist > :d0 OR (dist = :d0 AND image_id > :id0))] [AND image_id IN (...)]
    ORDER BY dist ASC, image_id ASC

and its COUNT(*), restated over tests/page_oracle.py; and the two kappa cuts of range_cut (page.cuh) restated in numpy
float32 / float64.  tests/test_range_args.py checks both against SQLite and the reference distance."""
import numpy as np

from tests import page_oracle


def answer(rows, ids, query, max_dist, cursor=None, allowed=None, dists=None):
    """(ids, dist, dot, norm2) of every row of the answer, in order; its length is the COUNT(*)."""
    ordered, dist = page_oracle.order(rows, ids, query, max_dist, allowed, dists)
    sel = page_oracle.after_cursor(ordered, ids, dist, cursor)
    dot, n2 = page_oracle.centred_terms(rows[sel], query)
    return ids[sel], dist[sel], dot, n2


# ---- the cuts --------------------------------------------------------------------------------------------------------
def certificate_margin(d: int) -> float:
    """api.cu certificate_margin: (4d + 3232) 2^-24, rounded to f32 and widened."""
    return float(np.float32((4.0 * d + 3232.0) * 2.0 ** -24))


def dist_bound(max_dist: float) -> np.float32:
    """api.cu dist_bound: the smallest f32 >= max_dist (NaN stays NaN)."""
    f = np.float32(max_dist)
    if float(f) < max_dist:
        f = np.nextafter(f, np.float32(np.inf))
    return f


def _f32_up(x: float) -> np.float32:
    f = np.float32(x)
    return np.nextafter(f, np.float32(np.inf)) if float(f) < x else f


def _f32_down(x: float) -> np.float32:
    f = np.float32(x)
    return np.nextafter(f, np.float32(-np.inf)) if float(f) > x else f


def range_cut(m: np.float32, margin: float):
    """(kappa_lo, kappa_in) of range_cut: kappa > kappa_in -> dist < m, kappa < kappa_lo -> dist >= m."""
    inf = np.float32(np.inf)
    m = np.float32(m)
    if np.isnan(m):
        return inf, inf
    if m > np.float32(999999.0):
        return -inf, -inf
    den = float(m) + 1.0
    if den <= 0.0:
        return inf, inf
    cs = 1.0 / den
    w = margin * max(1.0, cs)
    return _f32_down(cs - w), _f32_up(cs + w)


def kappas(rows, query):
    """The scan's ranking key of every row: fl(fl(fl(dot_i) * inv_norm_r) * inv_q), inverse norms rounded from f64."""
    cr = rows.astype(np.int64) * 2 - 255
    cq = query.astype(np.int64).ravel() * 2 - 255
    dot = cr @ cq
    inv_r = (1.0 / np.sqrt((cr * cr).sum(1).astype(np.float64))).astype(np.float32)
    inv_q = np.float32(1.0 / np.sqrt(float((cq * cq).sum())))
    return (dot.astype(np.float32) * inv_r) * inv_q
