// remove.cuh -- removal of rows by image id (pbx_corpus_remove): hole filling from the tail.
//
// With m rows removed out of n and n' = n - m, the j-th removed row below n' (in row order) receives the j-th surviving
// row at or above n' (in row order).  Only those rows move, sources (>= n') and destinations (< n') never overlap, and
// the layout is a pure function of the old layout and the request.  Steps, all on one stream:
//   mark_ids_kernel       one pass over the ids: a bit per row (binary search in the sorted request), the total m
//                         (filter.cuh, shared with the filtered searches)
//   remove_count_kernel   per 1024-row tile: holes below n', survivors at or above n'
//   remove_scan_kernel    exclusive scan of both counts over the tiles (one CTA)
//   remove_place_kernel   global rank of every hole / source (warp ballots inside the tile): the (hole, source) pairs
//   remove_move_kernel    pitch bytes per pair in 16-byte vectors, plus the id, inv_norm and row_sum of the row
// followed by block_meta_kernel (batch.cuh) over the blocks below n'.
#pragma once
#include "common.cuh"
#include "filter.cuh"

namespace pbx {

constexpr int kRemoveTileRows = kMarkTileRows;   // one CTA of 1024 threads, one row per thread

// A hole is a removed row below n_keep; a source is a surviving row at or above n_keep.
__device__ __forceinline__ void remove_roles(const uint32_t* __restrict__ flags, u64 row, u64 n, u64 n_keep, bool* hole, bool* src) {
    const bool in = row < n;
    const bool gone = in && ((flags[row >> 5] >> (row & 31)) & 1u);
    *hole = gone && row < n_keep;
    *src = in && !gone && row >= n_keep;
}

__global__ void __launch_bounds__(kRemoveTileRows) remove_count_kernel(const uint32_t* __restrict__ flags, u64 n, u64 n_keep,
                                                                       uint32_t* __restrict__ tile_holes, uint32_t* __restrict__ tile_srcs) {
    const u64 row = (u64)blockIdx.x * kRemoveTileRows + threadIdx.x;
    bool hole, src;
    remove_roles(flags, row, n, n_keep, &hole, &src);
    const int h = __syncthreads_count(hole);
    const int s = __syncthreads_count(src);
    if (threadIdx.x == 0) { tile_holes[blockIdx.x] = (uint32_t)h; tile_srcs[blockIdx.x] = (uint32_t)s; }
}

// In-place exclusive scan of a[0, n) and b[0, n) by one CTA of 1024 threads (each thread owns a contiguous run);
// *a_total = sum of a (the number of (hole, source) pairs).
__global__ void __launch_bounds__(1024) remove_scan_kernel(uint32_t* __restrict__ a, uint32_t* __restrict__ b, uint32_t n,
                                                           uint32_t* __restrict__ a_total) {
    __shared__ uint32_t wa[32], wb[32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t per = (n + 1023u) / 1024u;
    const uint32_t i0 = min(threadIdx.x * per, n), i1 = min(i0 + per, n);
    uint32_t sa = 0, sb = 0;
    for (uint32_t i = i0; i < i1; ++i) { sa += a[i]; sb += b[i]; }
    uint32_t ia = sa, ib = sb;                   // inclusive scan over the warp
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, ia, off), y = __shfl_up_sync(0xFFFFFFFFu, ib, off);
        if ((int)lane >= off) { ia += x; ib += y; }
    }
    if (lane == 31) { wa[warp] = ia; wb[warp] = ib; }
    __syncthreads();
    if (warp == 0) {
        const uint32_t va = wa[lane], vb = wb[lane];
        uint32_t xa = va, xb = vb;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, xa, off), y = __shfl_up_sync(0xFFFFFFFFu, xb, off);
            if ((int)lane >= off) { xa += x; xb += y; }
        }
        wa[lane] = xa - va; wb[lane] = xb - vb;
    }
    __syncthreads();
    uint32_t ra = wa[warp] + ia - sa, rb = wb[warp] + ib - sb;
    for (uint32_t i = i0; i < i1; ++i) {
        const uint32_t x = a[i], y = b[i];
        a[i] = ra; b[i] = rb;
        ra += x; rb += y;
    }
    if (threadIdx.x == 1023) *a_total = ra;     // the last thread's run ends at n
}

// hole_rows[j] / src_rows[j]: the j-th hole / source in row order (tile offsets from remove_scan_kernel).
__global__ void __launch_bounds__(kRemoveTileRows) remove_place_kernel(const uint32_t* __restrict__ flags, u64 n, u64 n_keep,
                                                                       const uint32_t* __restrict__ tile_holes, const uint32_t* __restrict__ tile_srcs,
                                                                       uint32_t* __restrict__ hole_rows, uint32_t* __restrict__ src_rows) {
    __shared__ uint32_t wh[32], ws[32];
    const u64 row = (u64)blockIdx.x * kRemoveTileRows + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    bool hole, src;
    remove_roles(flags, row, n, n_keep, &hole, &src);
    const uint32_t bh = __ballot_sync(0xFFFFFFFFu, hole), bs = __ballot_sync(0xFFFFFFFFu, src);
    if (lane == 0) { wh[warp] = __popc(bh); ws[warp] = __popc(bs); }
    __syncthreads();
    if (warp == 0) {
        const uint32_t vh = wh[lane], vs = ws[lane];
        uint32_t xh = vh, xs = vs;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t x = __shfl_up_sync(0xFFFFFFFFu, xh, off), y = __shfl_up_sync(0xFFFFFFFFu, xs, off);
            if ((int)lane >= off) { xh += x; xs += y; }
        }
        wh[lane] = xh - vh; ws[lane] = xs - vs;
    }
    __syncthreads();
    const uint32_t below = (1u << lane) - 1u;
    if (hole) hole_rows[tile_holes[blockIdx.x] + wh[warp] + __popc(bh & below)] = (uint32_t)row;
    if (src) src_rows[tile_srcs[blockIdx.x] + ws[warp] + __popc(bs & below)] = (uint32_t)row;
}

// One thread per (pair, 16-byte chunk); the chunk-0 thread also moves the row's id and metadata.  The number of pairs
// is read on the device (remove_scan_kernel wrote it): the host only knows its upper bound.
__global__ void remove_move_kernel(const uint32_t* __restrict__ hole_rows, const uint32_t* __restrict__ src_rows, const uint32_t* __restrict__ n_moves,
                                   uint32_t pitch16, uint4* __restrict__ rows, int64_t* __restrict__ ids, float* __restrict__ inv_norm,
                                   int* __restrict__ row_sum) {
    const u64 total = (u64)*n_moves * pitch16;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (u64)gridDim.x * blockDim.x) {
        const u64 j = t / pitch16;
        const uint32_t c = (uint32_t)(t - j * pitch16);
        const u64 dst = hole_rows[j], src = src_rows[j];
        rows[dst * pitch16 + c] = rows[src * pitch16 + c];
        if (c == 0) {
            ids[dst] = ids[src];
            inv_norm[dst] = inv_norm[src];
            row_sum[dst] = row_sum[src];
        }
    }
}

}  // namespace pbx
