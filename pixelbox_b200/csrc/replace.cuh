// replace.cuh -- replacement of the hashes of rows by image id, in place (pbx_corpus_replace).
//
// The host sorts the request: every listed id once, with the hash of its last occurrence, zero padded to the pitch (the
// row metadata sums run over the whole pitch).  Rows, ids and n do not change; a written row keeps its position.  Steps,
// all on one stream:
//   replace_mark_kernel        one pass over the ids (8 bytes per row): the lower bound of each row's id in the request; a
//                              (row, request index) pair per matching row, and the index of every 32-row block that holds
//                              one (a warp covers exactly one block), appended with one atomic per warp
//   replace_write_kernel       pitch bytes per pair in 16-byte vectors
//   replace_row_meta_kernel    inv_norm and row_sum of every written row (row_meta_warp, finalize.cuh)
//   replace_block_meta_kernel  the block metadata of every listed block (block_meta_warp, batch.cuh)
#pragma once
#include "common.cuh"
#include "filter.cuh"
#include "finalize.cuh"
#include "batch.cuh"

namespace pbx {

// counts[0] += matching rows, counts[1] += blocks that hold one.  Entries at or past `cap` are counted, not written: the
// host sizes the lists for one row per listed id and runs the pass again, with the exact size, when ids repeat in the corpus.
__global__ void __launch_bounds__(kMarkTileRows) replace_mark_kernel(const int64_t* __restrict__ ids, u64 n, const int64_t* __restrict__ req,
                                                                     u64 n_req, uint32_t cap, uint2* __restrict__ pairs,
                                                                     uint32_t* __restrict__ blocks, uint32_t* __restrict__ counts) {
    const u64 row = (u64)blockIdx.x * kMarkTileRows + threadIdx.x;
    u64 at = n_req;
    if (row < n) {
        const int64_t id = ids[row];
        at = sorted_lower_bound(req, n_req, id);
        if (at < n_req && req[at] != id) at = n_req;
    }
    const bool hit = at < n_req;
    const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, hit);
    if (ballot == 0) return;
    const uint32_t lane = threadIdx.x & 31;
    const int leader = __ffs(ballot) - 1;
    uint32_t base = 0, blk = 0;
    if ((int)lane == leader) {
        base = atomicAdd(counts, (uint32_t)__popc(ballot));
        blk = atomicAdd(counts + 1, 1u);
    }
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    if (hit) {
        const uint32_t slot = base + __popc(ballot & ((1u << lane) - 1u));
        if (slot < cap) pairs[slot] = make_uint2((uint32_t)row, (uint32_t)at);
    }
    if ((int)lane == leader && blk < cap) blocks[blk] = (uint32_t)(row >> 5);
}

// One thread per (pair, 16-byte chunk): row pairs[j].x receives request row pairs[j].y.
__global__ void replace_write_kernel(const uint2* __restrict__ pairs, u64 n_pairs, const uint4* __restrict__ src, uint32_t pitch16,
                                     uint4* __restrict__ rows) {
    const u64 total = n_pairs * pitch16;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (u64)gridDim.x * blockDim.x) {
        const u64 j = t / pitch16;
        const uint32_t c = (uint32_t)(t - j * pitch16);
        const uint2 p = pairs[j];
        rows[(u64)p.x * pitch16 + c] = src[(u64)p.y * pitch16 + c];
    }
}

// One warp per written row.
__global__ void replace_row_meta_kernel(const uint2* __restrict__ pairs, u64 n_pairs, const uint4* __restrict__ rows, uint32_t pitch16,
                                        uint32_t dim, float* __restrict__ inv_norm, int* __restrict__ row_sum) {
    const u64 j = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= n_pairs) return;
    row_meta_warp(rows, pitch16, dim, pairs[j].x, threadIdx.x & 31, inv_norm, row_sum);
}

// One warp per listed block.  A written row may lie outside its block's {norm, rowterm} range, which the batched epilogue
// trusts as a bound: the range of every block that holds one is recomputed.
__global__ void replace_block_meta_kernel(const uint32_t* __restrict__ blocks, u64 n_blocks, const float* __restrict__ inv_norm,
                                          const int* __restrict__ row_sum, uint32_t dim, u64 n_rows, float4* __restrict__ blk) {
    const u64 j = (u64)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (j >= n_blocks) return;
    block_meta_warp(inv_norm, row_sum, dim, blocks[j], threadIdx.x & 31, n_rows, blk);
}

}  // namespace pbx
