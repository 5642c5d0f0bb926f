// page.cuh -- the cut of a paged search (pbx_search_page and its twins): from each query's cursor (d0, id0), the kappa
// above which a row certainly sorts before the cursor (DESIGN.md section 5, "Paged searches").
//
// page_cut_kernel runs once per call, stream-ordered after the cursors are written, and reads them on the device: a
// pipeline can chain pages without a host read.  The search kernels then read one PageCut per query (common.cuh).
#pragma once
#include "common.cuh"
#include "../../include/pixelbox_b200.h"

namespace pbx {

// kappa_hi(d0), rounded up to f32.  With c* = 1/(d0 + 1) and the certificate margin M:
//   d0 NaN           -> every row sorts before the cursor (cut -inf, and d0 = +inf so that the replay drops any row)
//   d0 > 999999      -> every dist is <= 999999 < d0: cut -inf (d0 = +inf included)
//   d0 + 1 <= 0      -> no row is provably before the cursor: cut +inf (d0 <= -1, d0 = -inf; c* would be <= 0)
//   otherwise        -> c* + M * max(1, c*)
__device__ __forceinline__ PageCut page_cut(const pbx_hit& h, double margin) {
    PageCut pc;
    pc.id0 = h.image_id;
    pc.d0 = h.dist;
    pc.above = 0u;
    pc.pad = 0u;
    const float d0 = h.dist;
    if (d0 != d0) {
        pc.kappa_hi = -__int_as_float(0x7f800000);
        pc.d0 = __int_as_float(0x7f800000);
        pc.id0 = INT64_MAX;
    } else if (d0 > PBX_PLATEAU_DIST) {
        pc.kappa_hi = -__int_as_float(0x7f800000);
    } else {
        const double den = (double)d0 + 1.0;
        if (den <= 0.0) {
            pc.kappa_hi = __int_as_float(0x7f800000);
        } else {
            const double cs = 1.0 / den;
            pc.kappa_hi = __double2float_ru(cs + margin * fmax(1.0, cs));
        }
    }
    return pc;
}

// The two cuts of a range search (range.cuh) for the f32 bound m = dist_bound(max_dist), with c* = 1/(m + 1) and the
// certificate margin M (DESIGN.md section 5, "Range searches"):
//   kappa > kappa_in  ->  dist < m  (certainly inside: page_cut's kappa_hi(m), rounded up)
//   kappa < kappa_lo  ->  dist >= m (certainly outside: c* - M * max(1, c*), rounded down)
//   m NaN            -> no row is inside: both +inf
//   m > 999999       -> every dist is <= 999999 < m: both -inf
//   m + 1 <= 0       -> every dist is > -1 >= m: both +inf
struct RangeCut {
    float kappa_lo, kappa_in;
};
__device__ __forceinline__ RangeCut range_cut(float m, double margin) {
    const float inf = __int_as_float(0x7f800000);
    RangeCut rc;
    if (m != m) {
        rc.kappa_lo = inf; rc.kappa_in = inf;
    } else if (m > PBX_PLATEAU_DIST) {
        rc.kappa_lo = -inf; rc.kappa_in = -inf;
    } else {
        const double den = (double)m + 1.0;
        if (den <= 0.0) {
            rc.kappa_lo = inf; rc.kappa_in = inf;
        } else {
            const double cs = 1.0 / den, w = margin * fmax(1.0, cs);
            rc.kappa_in = __double2float_ru(cs + w);
            rc.kappa_lo = __double2float_rd(cs - w);
        }
    }
    return rc;
}

__global__ void page_cut_kernel(const pbx_hit* __restrict__ after, uint32_t nq, double margin, PageCut* __restrict__ out) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) out[q] = page_cut(after[q], margin);
}

}  // namespace pbx
