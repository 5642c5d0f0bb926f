"""Complete reference of searches over a synthetic corpus (`Corpus.fill_synthetic(n, seed, first_row)`), at any size.

The corpus is never read through the library: its rows are regenerated from the definition in pixelbox_b200/synth.py
with torch (on the GPU at scale), in chunks, and scored exactly:

* cos* = dot / sqrt(n_q n_r), dot = sum c(q) c(r), n = sum c(.)^2, c(v) = 2v - 255.  The centred values are small
  integers, so a float64 matmul gives dot and n exactly (whatever TF32 or emulation settings are in force); cos* is
  then computed in float64.
* For each query let c_K be the K-th largest cos* among the eligible rows.  Every row the reference's f32
  cosine_distance could rank among the first K has cos* >= c_K - M, with M = (4d + 3232) 2^-24 the margin of the
  search's certificate (DESIGN.md §5): |cos_ref - cos*| <= eps_d for every row, and M > 2 eps_d + 2^-22.  So the rows of
  that band are the only candidates; their bytes are regenerated on the host and oracle.topk ranks them, which gives
  ids, dist bits, dot and norm2 of the answer.

Eligible rows: not removed, not replaced (the replaced and appended rows come from a small host overlay that is scored
the same way), and inside the INCLUDE set or outside the EXCLUDE set of the call.  A page is a slice of one deep top-K,
so no cursor logic is needed here.
"""
from __future__ import annotations

import numpy as np
import torch

from oracle import oracle

_MASK64 = (1 << 64) - 1


def _s64(v: int) -> int:
    """A uint64 constant as the int64 with the same bits."""
    v &= _MASK64
    return v - (1 << 64) if v >= 1 << 63 else v


_GOLDEN = _s64(0x9E3779B97F4A7C15)
_MIX1 = _s64(0xBF58476D1CE4E5B9)
_MIX2 = _s64(0x94D049BB133111EB)
_ROWMUL = _s64(0xD1342543DE82EF95)


def _srl(z: torch.Tensor, s: int) -> torch.Tensor:
    """Logical right shift of int64 bits: the arithmetic shift with the sign-extended bits masked off."""
    return (z >> s) & ((1 << (64 - s)) - 1)


def _splitmix64(z: torch.Tensor) -> torch.Tensor:
    z = z + _GOLDEN                               # int64 add and multiply wrap around: the uint64 arithmetic of synth.py
    z = (z ^ _srl(z, 30)) * _MIX1
    z = (z ^ _srl(z, 27)) * _MIX2
    return z ^ _srl(z, 31)


def _gen(rows: torch.Tensor, seed: int, dim: int) -> torch.Tensor:
    """uint8 [len(rows), dim]: the synthetic rows at these global row indices (int64 tensor, any device)."""
    chunks = (dim + 7) // 8
    rk = _splitmix64(rows * _ROWMUL ^ _s64(seed))
    x = _splitmix64(rk[:, None] + torch.arange(chunks, dtype=torch.int64, device=rows.device)[None, :])
    # byte b of chunk c is byte b (little endian) of x: the bytes of the int64 tensor as they lie in memory
    return x.contiguous().view(torch.uint8).reshape(rows.numel(), chunks * 8)[:, :dim]


def synth_rows_torch(seed: int, first_row: int, nrows: int, dim: int, device="cpu") -> torch.Tensor:
    """Rows [first_row, first_row + nrows) of the synthetic corpus as uint8 [nrows, dim] on `device`."""
    rows = torch.arange(nrows, dtype=torch.int64, device=device) + _s64(first_row)
    return _gen(rows, seed, dim).contiguous()


def margin(dim: int) -> float:
    """M = (4d + 3232) 2^-24, the certificate margin of DESIGN.md §5."""
    return (4 * dim + 3232) * 2.0 ** -24


def _in_sorted(values: torch.Tensor, sorted_set: torch.Tensor) -> torch.Tensor:
    if sorted_set.numel() == 0:
        return torch.zeros_like(values, dtype=torch.bool)
    i = torch.searchsorted(sorted_set, values).clamp_(max=sorted_set.numel() - 1)
    return sorted_set[i] == values


def _sorted_ids(ids, device) -> torch.Tensor:
    a = np.unique(np.asarray(ids, dtype=np.int64).reshape(-1))
    return torch.from_numpy(a).to(device)


class SynthReference:
    """The answers of searches over `fill_synthetic(n, seed, first_row)` on a corpus of `dim`, after the mutations
    recorded with remove / set_rows.  Image id of synthetic row r (local) is first_row + r + 1."""

    def __init__(self, n: int, seed: int, dim: int, first_row: int = 0, device="cpu", chunk_bytes: int = 4 << 30):
        self.n, self.seed, self.dim, self.first_row = int(n), int(seed), int(dim), int(first_row)
        self.device = torch.device(device)
        self.chunk_bytes = int(chunk_bytes)         # float64 scratch of one chunk: centred rows + scores
        self.removed = np.zeros(0, np.int64)
        self.overlay = {}                           # image id -> row bytes (replaced or appended rows)

    # -- the table's mutations ----------------------------------------------------------------
    def remove(self, ids) -> None:
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        self.removed = np.union1d(self.removed, ids)
        for i in ids.tolist():
            self.overlay.pop(int(i), None)

    def set_rows(self, ids, rows) -> None:
        """Replaced rows (ids of synthetic rows) and appended rows (new ids): their bytes from now on."""
        rows = np.asarray(rows, dtype=np.uint8).reshape(-1, self.dim)
        for i, r in zip(np.asarray(ids, dtype=np.int64).tolist(), rows):
            self.overlay[int(i)] = r.copy()
        self.removed = np.setdiff1d(self.removed, np.asarray(ids, dtype=np.int64))

    def row_bytes(self, ids) -> np.ndarray:
        """The current bytes of the rows with these image ids (host, [len(ids), dim])."""
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        over = np.isin(ids, np.fromiter(self.overlay, np.int64, len(self.overlay)))
        syn = ids[~over]
        assert np.all((syn > self.first_row) & (syn <= self.first_row + self.n)), "an id that is no row of the corpus"
        out = np.zeros((ids.size, self.dim), np.uint8)
        out[~over] = _gen(torch.from_numpy(syn - 1).to(self.device), self.seed, self.dim).cpu().numpy()
        for j in np.nonzero(over)[0].tolist():
            out[j] = self.overlay[int(ids[j])]
        return out

    # -- the reference ------------------------------------------------------------------------
    def _scores(self, rows_u8: torch.Tensor, cq: torch.Tensor, inv_sqrt_nq: torch.Tensor) -> torch.Tensor:
        cr = rows_u8.to(torch.float64) * 2 - 255
        dot = cq @ cr.T                                     # exact: |values| < 2^53
        nr = (cr * cr).sum(dim=1)
        return dot * inv_sqrt_nq[:, None] / torch.sqrt(nr)[None, :]

    def topk(self, queries, k: int, max_dist: float = 1e3, include=None, exclude=None):
        """Per query (ids, dist, dot, norm2) of the first k rows by (dist, image_id) with dist < max_dist: the search's
        answer, bit for bit.  k may exceed PBX_MAX_K (a page is a slice of this)."""
        assert max_dist <= 1e3, "the band argument needs the plateau out of reach"
        assert include is None or exclude is None
        queries = np.ascontiguousarray(np.asarray(queries, dtype=np.uint8).reshape(-1, self.dim))
        nq, dev = queries.shape[0], self.device
        cap = 10 * k + 1000                                 # the band may not be larger than this
        cq = torch.from_numpy(queries).to(dev).to(torch.float64) * 2 - 255
        inv_sqrt_nq = 1.0 / torch.sqrt((cq * cq).sum(dim=1))
        removed = _sorted_ids(np.concatenate([self.removed, np.fromiter(self.overlay, np.int64, len(self.overlay))]), dev)
        inc = None if include is None else _sorted_ids(include, dev)
        exc = None if exclude is None else _sorted_ids(exclude, dev)

        best_v = torch.empty((nq, 0), dtype=torch.float64, device=dev)
        best_i = torch.empty((nq, 0), dtype=torch.int64, device=dev)
        total = 0

        def take(scores: torch.Tensor, ids: torch.Tensor):
            nonlocal best_v, best_i, total
            total += scores.shape[1]
            v, j = torch.topk(scores, min(cap, scores.shape[1]), dim=1, sorted=False)
            v, i = torch.cat([best_v, v], dim=1), torch.cat([best_i, ids[j]], dim=1)
            v, j = torch.topk(v, min(cap, v.shape[1]), dim=1, sorted=True)
            best_v, best_i = v, torch.gather(i, 1, j)

        chunk_rows = max(1024, self.chunk_bytes // (8 * (self.dim + nq + 2)))
        for r0 in range(0, self.n, chunk_rows):
            m = min(chunk_rows, self.n - r0)
            ids = torch.arange(m, dtype=torch.int64, device=dev) + (self.first_row + r0 + 1)
            keep = ~_in_sorted(ids, removed)
            if inc is not None:
                keep &= _in_sorted(ids, inc)
            if exc is not None:
                keep &= ~_in_sorted(ids, exc)
            if not bool(keep.any()):
                continue
            if not bool(keep.all()):
                ids = ids[keep]
            rows = _gen(ids - 1, self.seed, self.dim)
            take(self._scores(rows, cq, inv_sqrt_nq), ids)
        o_ids = np.fromiter(self.overlay, np.int64, len(self.overlay))
        if include is not None:
            o_ids = o_ids[np.isin(o_ids, np.asarray(include, dtype=np.int64))]
        if exclude is not None:
            o_ids = o_ids[~np.isin(o_ids, np.asarray(exclude, dtype=np.int64))]
        if o_ids.size:
            o_rows = torch.from_numpy(np.stack([self.overlay[int(i)] for i in o_ids])).to(dev)
            take(self._scores(o_rows, cq, inv_sqrt_nq), torch.from_numpy(o_ids).to(dev))

        best_v, best_i = best_v.cpu().numpy(), best_i.cpu().numpy()
        M = margin(self.dim)
        bands = []
        for qi in range(nq):
            if total <= k:                                  # every eligible row is a candidate
                bands.append(best_i[qi])
                continue
            ck = best_v[qi, k - 1]
            assert ck - M > 2e-6, f"query {qi}: the band reaches the plateau (c_k = {ck})"
            inband = best_v[qi] >= ck - M
            assert inband.sum() < best_v.shape[1] or total <= cap, \
                f"query {qi}: more than {cap} rows within the margin of the {k}-th best (degenerate corpus?)"
            bands.append(best_i[qi][inband])
        cand = np.unique(np.concatenate(bands))
        cand_rows = self.row_bytes(cand)
        out = []
        for qi, band in enumerate(bands):
            rows = cand_rows[np.searchsorted(cand, band)]
            out.append(oracle.topk(rows, band, queries[qi], k, max_dist))
        return out
