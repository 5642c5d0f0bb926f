// range_sort.cu -- the radix sorts of a range search (range.cuh), CUB's DeviceRadixSort.  A translation unit of its own:
// CUB's kernels and their shared memory stay out of api.cu, whose kernels compile exactly as without them.
// (The declarations are in range.cuh, which this file does not include: its kernels are api.cu's.)
#include <cub/device/device_radix_sort.cuh>
#include <stdint.h>

namespace pbx {

typedef unsigned long long u64;

cudaError_t range_sort_pairs(void* tmp, size_t& tmp_bytes, const u64* keys_in, u64* keys_out, const uint32_t* vals_in,
                             uint32_t* vals_out, uint32_t n, cudaStream_t s) {
    return cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys_in, keys_out, vals_in, vals_out, n, 0, 64, s);
}

cudaError_t range_sort_pairs(void* tmp, size_t& tmp_bytes, const uint32_t* keys_in, uint32_t* keys_out, const uint32_t* vals_in,
                             uint32_t* vals_out, uint32_t n, cudaStream_t s) {
    return cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys_in, keys_out, vals_in, vals_out, n, 0, 32, s);
}

}  // namespace pbx
