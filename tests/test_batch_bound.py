"""The batched epilogue's selection bound, restated in numpy float32 (pixelbox_b200/csrc/batch.cuh: batch_bound_t4,
batch_bound_cq, `bound`, block_meta_kernel, row_meta_kernel, batch_prep_kernel) and checked for the one property the
whole path relies on: a row that passes the exact test  fl(fl(dot_i) * inv_norm_r) >= thr  has a raw score
S = sum (q_i - 128) r_i  at or above the block's integer bound v -- a bound that is too tight drops a true neighbour
without any certificate noticing (the certificate only sees candidates that were found).  CPU only."""
import numpy as np
import pytest

f32 = np.float32


def block_case(rng, d, kind):
    """32 corpus rows + a query of a given flavour."""
    if kind == "uniform":
        rows = rng.integers(0, 256, size=(32, d))
    elif kind == "wild":        # almost no norm, maximal norm, dark and ordinary rows in one block
        rows = rng.integers(0, 256, size=(32, d))
        rows[0:8] = rng.integers(127, 129, size=(8, d))
        rows[8:16] = rng.integers(0, 2, size=(8, d)) * 255
        rows[16:24] = rng.integers(0, 40, size=(8, d))
    else:                       # "near": small perturbations of one row
        rows = np.clip(rng.integers(0, 256, size=(1, d)) + rng.integers(-3, 4, size=(32, d)), 0, 255)
    q = rng.integers(0, 256, size=d)
    if rng.random() < 0.5:
        q = np.clip(rows[rng.integers(0, 32)] + rng.integers(-10, 11, size=d), 0, 255)
    if rng.random() < 0.3:
        q = 255 - q             # anti-correlated: negative cosines, negative thresholds
    return rows.astype(np.int64), q.astype(np.int64)


def bound_and_scores(rows, q, thr):
    d = rows.shape[1]
    c = 2 * rows - 255
    n2 = (c * c).sum(1)
    inv = (1.0 / np.sqrt(n2.astype(np.float64))).astype(f32)                 # row_meta_kernel
    rt = 2 * rows.sum(1) - 255 * d                                            # rowterm
    norm_lo = f32(1.0) / inv.max()                                            # block_meta_kernel: __fdiv_rn(1, inv_hi)
    norm_hi = f32(1.0) / inv.min()
    z = f32(0.25) * f32(rt.max())
    qs = q - 128
    S = (qs[None, :] * rows).sum(1)                                           # the tensor cores' s8 x u8 -> s32
    ct = -510 * int(qs.sum())                                                 # batch_prep_kernel
    dot = 4 * S + rt + ct
    assert np.array_equal(dot, ((2 * q - 255)[None, :] * c).sum(1))           # the integer identity of DESIGN section 3
    kf = dot.astype(f32) * inv                                                # fl(fl(dot_i) * inv_r), both in f32
    thr = f32(thr)
    t4 = f32(0.25) * thr * (f32(1.0) - f32(5.0e-6) if thr >= 0 else f32(1.0) + f32(5.0e-6))      # batch_bound_t4
    cf = f32(ct)
    cq = f32(-0.25) * cf - (f32(1.0e-6) * abs(cf) + f32(8.0))                 # batch_bound_cq
    nsel = norm_lo if t4 >= 0 else norm_hi
    fma = f32(np.float64(t4) * np.float64(nsel) + np.float64(cq))             # fmaf: one rounding (f64 holds the product exactly)
    v = int(np.floor(np.float64(fma - z)))
    return S, kf, thr, v


@pytest.mark.parametrize("d", [32, 64, 256, 1024])
@pytest.mark.parametrize("kind", ["uniform", "wild", "near"])
def test_bound_never_excludes_a_passing_row(d, kind):
    rng = np.random.default_rng([d, ["uniform", "wild", "near"].index(kind)])     # not hash(): it changes with PYTHONHASHSEED
    checked = 0
    for _ in range(120):
        rows, q = block_case(rng, d, kind)
        S, kf, _, _ = bound_and_scores(rows, q, 0.0)
        # thresholds exactly at, just below and just above the kappa' of some rows (the boundary is where a bound breaks),
        # plus a few far away on both sides
        cands = list(kf[rng.integers(0, 32, 4)])
        thrs = [t for k in cands for t in (k, np.nextafter(k, f32(-np.inf)), np.nextafter(k, f32(np.inf)))]
        thrs += [f32(0.0), f32(-1.0e30), kf.min() - f32(1.0), kf.max() * f32(0.5)]
        for thr in thrs:
            S, kf, t, v = bound_and_scores(rows, q, thr)
            passing = kf >= t
            # (v - 1: the numpy fmaf above may differ from the GPU's by one unit in the last place in rare double roundings)
            assert np.all(S[passing] >= v - 1), (d, kind, float(t), int(v), S[passing].min())
            checked += int(passing.sum())
    assert checked > 500


def test_bound_is_not_vacuous():
    """... and it does prune: on uniform random blocks at a threshold four sigma up, almost no block passes."""
    rng = np.random.default_rng(5)
    d, passes = 256, 0
    for _ in range(400):
        rows, q = block_case(rng, d, "uniform")
        q = rng.integers(0, 256, size=d).astype(np.int64)
        S, kf, t, v = bound_and_scores(rows, q, np.float32(0.27 * np.sqrt(float(((2 * q - 255) ** 2).sum()))))
        passes += int(S.max() >= v)
    assert passes <= 8
