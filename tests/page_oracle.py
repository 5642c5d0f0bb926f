"""Page oracle of the paged searches: the keyset SQL

    SELECT ... WHERE dist < :max_dist AND (dist > :d0 OR (dist = :d0 AND image_id > :id0)) [AND image_id IN (...)]
    ORDER BY dist ASC, image_id ASC LIMIT :k

restated in numpy over oracle.all_distances (the reference's f32 cosine_distance, bit for bit).  tests/test_page_args.py
checks it against that SQL in SQLite."""
import numpy as np

from oracle import oracle


def centred_terms(rows: np.ndarray, query: np.ndarray):
    """(dot, norm2) of rows against the query: sum c(q) c(r) and sum c(r)^2 with c(v) = 2v - 255, exact in int64."""
    cr = rows.astype(np.int64) * 2 - 255
    cq = query.astype(np.int64).ravel() * 2 - 255
    return (cr @ cq).astype(np.int32), (cr * cr).sum(axis=1).astype(np.int32)


def order(rows, ids, query, max_dist, allowed=None, dists=None):
    """Row indices of every row with dist < max_dist (and allowed), ordered by (dist, image_id), and the dists."""
    dist = oracle.all_distances(rows, query) if dists is None else dists
    mask = dist.astype(np.float64) < float(max_dist)
    if allowed is not None:
        mask &= allowed
    idx = np.nonzero(mask)[0]
    return idx[np.lexsort((ids[idx], dist[idx]))], dist


def after_cursor(ordered, ids, dist, cursor):
    """The suffix of `ordered` that sorts strictly after cursor (d0, id0); None: all of it."""
    if cursor is None:
        return ordered
    d0, id0 = np.float32(cursor[0]), np.int64(cursor[1])
    if np.isnan(d0):
        return ordered[:0]
    dd, ii = dist[ordered], ids[ordered]
    return ordered[(dd > d0) | ((dd == d0) & (ii > id0))]


def page(rows, ids, query, k, max_dist, cursor=None, allowed=None, dists=None):
    """(ids, dist, dot, norm2) of the k rows after `cursor`: what the keyset SQL returns."""
    ordered, dist = order(rows, ids, query, max_dist, allowed, dists)
    sel = after_cursor(ordered, ids, dist, cursor)[:k]
    dot, n2 = centred_terms(rows[sel], query)
    return ids[sel], dist[sel], dot, n2
