// filter.cuh -- one bit per row from a set of image ids: the mark pass of pbx_corpus_remove (rows to remove) and of the
// filtered searches (rows a search may return, pbx_search_filtered and its twins).  pbx_corpus_replace's mark pass
// (replace.cuh) uses the same binary search.
//
// mark_ids_kernel is one pass over the row ids (8 bytes per row) with a binary search of each id in the sorted set; the
// search kernels then test bit (row & 31) of word row >> 5 (row_allowed, common.cuh).
#pragma once
#include "common.cuh"

namespace pbx {

constexpr int kMarkTileRows = 1024;          // one CTA of 1024 threads, one row per thread

// Binary search in an ascending set (duplicates allowed): the first index whose element is not below v (n_set if none).
// v is in the set iff the result is < n_set and holds v.  Any input is memory-safe: an unsorted set gives a wrong
// answer, never an out-of-bounds read.
__device__ __forceinline__ u64 sorted_lower_bound(const int64_t* __restrict__ set, u64 n_set, int64_t v) {
    u64 lo = 0, hi = n_set;
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if (set[mid] < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// flags[w] bit l: row 32 w + l (< n) has its id in the set, or with `invert` has not.  *marked += number of set bits.
// Words are written for rows < n only; bits of rows >= n in the last word are 0.
__global__ void __launch_bounds__(kMarkTileRows) mark_ids_kernel(const int64_t* __restrict__ ids, u64 n, const int64_t* __restrict__ set,
                                                                 u64 n_set, uint32_t invert, uint32_t* __restrict__ flags, u64* __restrict__ marked) {
    const u64 row = (u64)blockIdx.x * kMarkTileRows + threadIdx.x;
    bool bit = false;
    if (row < n) {
        const int64_t id = ids[row];
        const u64 at = sorted_lower_bound(set, n_set, id);
        bit = (at < n_set && set[at] == id) != (invert != 0);
    }
    const uint32_t word = __ballot_sync(0xFFFFFFFFu, bit);
    if ((threadIdx.x & 31) == 0 && row < n) flags[row >> 5] = word;
    const int cnt = __syncthreads_count(bit);
    if (threadIdx.x == 0 && cnt) atomicAdd(marked, (u64)cnt);
}

// Device-resident filters must be sorted ascending: *unsorted = 1 if set[i - 1] > set[i] for some i (the word is zeroed
// by the host beforehand).  Stream-ordered, no host synchronisation.
__global__ void ids_unsorted_kernel(const int64_t* __restrict__ set, u64 n_set, uint32_t* __restrict__ unsorted) {
    for (u64 i = 1 + (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_set; i += (u64)gridDim.x * blockDim.x)
        if (set[i - 1] > set[i]) { *unsorted = 1u; return; }
}

// After the search of an unsorted device filter: every count becomes PBX_COUNT_FILTER_UNSORTED (the hits are not valid).
__global__ void filter_unsorted_count_kernel(const uint32_t* __restrict__ unsorted, uint32_t* __restrict__ count, uint32_t nq, uint32_t marker) {
    if (*unsorted == 0) return;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += gridDim.x * blockDim.x) count[i] = marker;
}

}  // namespace pbx
