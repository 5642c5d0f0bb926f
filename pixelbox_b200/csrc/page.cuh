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

__global__ void page_cut_kernel(const pbx_hit* __restrict__ after, uint32_t nq, double margin, PageCut* __restrict__ out) {
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) out[q] = page_cut(after[q], margin);
}

}  // namespace pbx
