// view.cuh -- views of a corpus (pbx_corpus_view_create): a corpus holding a copy of the parent's rows whose image id is
// in a set, kept current by the parent's mutating calls.
//
// Collecting the rows of a parent range [r0, r1) into a view, all on one stream:
//   mark_ids_kernel       one pass over the range's ids against the view's sorted set (filter.cuh)
//   remove_count_kernel   \  compaction of the bitmap into ascending row indices: remove.cuh's count / scan / place with
//   remove_scan_kernel     > n_keep = the range size, so every marked row is a "hole" and there are no sources; the j-th
//   remove_place_kernel   /  hole is the j-th marked row of the range
//   view_gather_kernel    pitch bytes per row in 16-byte vectors, plus the id, inv_norm and row_sum, behind the view's rows
// followed by block_meta_kernel (batch.cuh) over the view blocks the new rows touch.  Removal and replacement on a view are
// pbx_corpus_remove's and pbx_corpus_replace's own code.
#pragma once
#include "common.cuh"
#include "filter.cuh"
#include "remove.cuh"

namespace pbx {

// One thread per (row, 16-byte chunk): parent row src0 + src_rows[j] becomes view row dst0 + j, j < n_rows.  The chunk-0
// thread also copies the id and the row metadata: copied, not recomputed, so they are the parent's bit for bit.
__global__ void view_gather_kernel(const uint32_t* __restrict__ src_rows, u64 n_rows, u64 src0, uint32_t pitch16,
                                   const uint4* __restrict__ p_rows, const int64_t* __restrict__ p_ids, const float* __restrict__ p_inv,
                                   const int* __restrict__ p_rsum, u64 dst0, uint4* __restrict__ v_rows, int64_t* __restrict__ v_ids,
                                   float* __restrict__ v_inv, int* __restrict__ v_rsum) {
    const u64 total = n_rows * pitch16;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (u64)gridDim.x * blockDim.x) {
        const u64 j = t / pitch16;
        const uint32_t c = (uint32_t)(t - j * pitch16);
        const u64 src = src0 + src_rows[j], dst = dst0 + j;
        v_rows[dst * pitch16 + c] = p_rows[src * pitch16 + c];
        if (c == 0) {
            v_ids[dst] = p_ids[src];
            v_inv[dst] = p_inv[src];
            v_rsum[dst] = p_rsum[src];
        }
    }
}

}  // namespace pbx
