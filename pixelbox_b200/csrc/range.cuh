// range.cuh -- range searches (pbx_search_range): every row with dist < max_dist, and its exact count, in one streaming
// pass over the shard.  The query without its LIMIT:
//     SELECT image_id, cosine_distance(?, hash) AS dist FROM semantic_hashes WHERE dist < ? ORDER BY dist ASC
//
// 1. range_scan_kernel: the scan's stream (same lane layouts, dp2a dot, transposing butterfly, warp-autonomous chunk
//    claims) without thresholds or top-k buffers.  range_cut (page.cuh) splits kappa into three bands: below kappa_lo a
//    row is certainly outside, above kappa_in certainly inside, in between only the replay can tell.  Every allowed row
//    at or below the cursor cut with kappa >= kappa_lo is appended as (row, kappa) to a global candidate buffer: one
//    ballot per warp iteration into a per-warp stage in shared memory, one atomic per flush of the stage.  In count-only
//    mode the rows that are certainly inside (and certainly after the cursor) are counted instead of appended.  The
//    counter runs past the buffer's capacity: the host reads it, grows the buffer and runs the pass again when it
//    overflowed.
// 2. range_replay_kernel: one thread per candidate, the bit-exact replay of the reference's f32 arithmetic
//    (replay_row<true>: dist, dot and norm2); rows with dist >= max_dist or at or before the cursor are dropped.  Full
//    mode writes a (dist, image_id) sort key and the record of every candidate (a dropped one sorts last); count-only
//    mode counts the survivors.
// 3. The records are ordered by (dist, image_id) with two stable radix sorts (image_id, then dist; range_sort.cu) and
//    range_gather_kernel writes the first rows out.
#pragma once
#include "scan.cuh"
#include "page.cuh"

namespace pbx {

// counters of one range pass (device words, zeroed before the scan)
enum : uint32_t { kRangeTile = 0, kRangeCand = 1, kRangeDirect = 2, kRangeHits = 3, kRangeCounters = 4 };

struct RangeScanParams {
    const uint4* rows;          // [capacity][pitch16]
    const float* inv_norm;
    uint32_t n;
    uint32_t pitch16;
    const int16_t* q16;         // [pitch] centred query
    const QueryHeader* qh;
    const uint32_t* allow;      // filter bitmap (NULL: every row)
    const PageCut* cut;         // cursor (NULL: none)
    float m;                    // dist_bound(max_dist)
    uint32_t count_only;
    double margin;              // certificate margin M
    uint2* cand;                // [cand_cap] (row, kappa bits)
    uint32_t cand_cap;
    uint32_t* counters;         // [kRangeCounters]
};

// Fast shapes: pitch16 == L * C.  RAGGED: any pitch16 <= L * C, row stride at run time.  L, C and MINB as scan_kernel's.
template <int L, int C, bool RAGGED, int MINB>
__global__ void __launch_bounds__(kScanThreads, MINB)
range_scan_kernel(const RangeScanParams p) {
    constexpr int G = 32 / L;
    constexpr int P16 = L * C;
    const uint32_t PR = RAGGED ? p.pitch16 : (uint32_t)P16;
    const int lane = threadIdx.x & 31;
    const int g = lane / L, j = lane % L;

    int q[C][8];
    uint32_t coff[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const bool has = !RAGGED || (uint32_t)(j + c * L) < PR;
        coff[c] = has ? (uint32_t)(j + c * L) : PR - 1u;
        const int4* src = reinterpret_cast<const int4*>(p.q16 + (size_t)(has ? (j + c * L) : 0) * 16);
        int4 a = __ldg(src), b = __ldg(src + 1);
        if (!has) { a = make_int4(0, 0, 0, 0); b = a; }
        q[c][0] = a.x; q[c][1] = a.y; q[c][2] = a.z; q[c][3] = a.w;
        q[c][4] = b.x; q[c][5] = b.y; q[c][6] = b.z; q[c][7] = b.w;
    }
    const QueryHeader qh = *p.qh;
    const int bias = -255 * qh.sum_cq;
    const float inf = __int_as_float(0x7f800000);
    const float cut = page_kappa_hi(p.cut);
    const RangeCut rc = range_cut(p.m, p.margin);
    // count-only: a row is counted without a replay when it is certainly inside (kappa > kappa_in) and certainly after
    // the cursor: kappa < kappa_lo of the next f32 above d0 means dist > d0
    float k_in = inf, k_after = inf;
    if (p.count_only) {
        k_in = rc.kappa_in;
        if (p.cut) k_after = range_cut(nextafterf(p.cut->d0, inf), p.margin).kappa_lo;
    }

    // appended rows are staged per warp in shared memory and written out with one atomic per flush: the flush comes when
    // another chunk might not fit, so a dense answer costs one atomic per ~kChunkRows rows, not one per warp iteration
    __shared__ uint2 stage[kScanWarps][2 * kChunkRows];
    uint2* const st = stage[threadIdx.x >> 5];
    uint32_t n_st = 0;                                  // warp-uniform
    auto flush = [&]() {
        __syncwarp();
        uint32_t at = 0;
        if (lane == 0) at = atomicAdd(p.counters + kRangeCand, n_st);
        at = __shfl_sync(0xFFFFFFFFu, at, 0);
        for (uint32_t i = lane; i < n_st; i += 32)
            if (at + i < p.cand_cap) p.cand[at + i] = st[i];
        __syncwarp();
        n_st = 0;
    };

    constexpr uint32_t GRAB = (P16 >= 16) ? 1u : 16u / P16;
    const uint32_t n_chunks = (p.n + kChunkRows - 1) / kChunkRows;
    uint32_t cur = 0, end = 0, nxt = 0, direct = 0;
    if (lane == 0) nxt = atomicAdd(p.counters + kRangeTile, GRAB);
    for (;;) {
        if (cur == end) {
            cur = __shfl_sync(0xFFFFFFFFu, nxt, 0);
            end = cur + GRAB;
            if (lane == 0 && cur < n_chunks) nxt = atomicAdd(p.counters + kRangeTile, GRAB);
        }
        if (cur >= n_chunks) break;
        const uint32_t chunk_row0 = cur * kChunkRows;
        ++cur;
        constexpr int UNR = (L * C >= 16) ? 1 : kItersPerChunk;
#pragma unroll UNR
        for (int it = 0; it < kItersPerChunk; ++it) {
            const uint32_t row0 = chunk_row0 + (uint32_t)it * kRowsPerWarpIter;
            const uint32_t my_row = row0 + (uint32_t)(j * G + g);
            const uint32_t allow_word = p.allow ? __ldg(p.allow + (row0 >> 5)) : ~0u;
            const float inv_r = __ldg(p.inv_norm + my_row);
            const uint4* base = p.rows + (size_t)row0 * PR + (size_t)g * PR + (RAGGED ? 0 : j);
            int acc[L];
#pragma unroll
            for (int r = 0; r < L; ++r) {
                int a = 0;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    uint4 v = ldg_stream(base + (size_t)(r * G) * PR + (RAGGED ? coff[c] : (uint32_t)(c * L)));
                    a = dot16(v, q[c], a);
                }
                acc[r] = a;
            }
            const int s = transpose_reduce<L>(acc, j);
            const float kappa = __fmul_rn(__fmul_rn((float)(2 * s + bias), inv_r), qh.inv_q);
            const bool live = my_row < p.n && ((allow_word >> (my_row & 31u)) & 1u) && kappa <= cut;
            const bool inside = live && kappa > k_in && kappa < k_after;
            const bool push = live && !inside && kappa >= rc.kappa_lo;
            direct += __popc(__ballot_sync(0xFFFFFFFFu, inside));
            const unsigned mask = __ballot_sync(0xFFFFFFFFu, push);
            if (push) st[n_st + __popc(mask & ((1u << lane) - 1u))] = make_uint2(my_row, __float_as_uint(kappa));
            n_st += __popc(mask);
        }
        if (n_st > kChunkRows) flush();
    }
    if (n_st) flush();
    if (lane == 0 && direct) atomicAdd(p.counters + kRangeDirect, direct);
}

struct RangeReplayParams {
    const uint8_t* rows;        // [capacity][pitch]
    const int64_t* ids;
    uint32_t pitch, dim;
    const uint8_t* qbytes;      // [pitch] raw query bytes
    const int16_t* q16;
    const QueryHeader* qh;
    const PageCut* cut;
    float m;
    uint32_t n_cand;
    const uint2* cand;
    uint32_t* counters;         // counters[kRangeHits] += the surviving candidates
    // full mode (NULL in count-only mode): one sort key pair, index and record per candidate
    uint32_t* key_dist;         // ord(dist), ~0 for a dropped row
    u64* key_id;                // image_id with its sign bit flipped (ascending as unsigned)
    uint32_t* index;
    pbx_hit* recs;
};

constexpr int kRangeReplayThreads = 256;

__global__ void __launch_bounds__(kRangeReplayThreads)
range_replay_kernel(const RangeReplayParams p) {
    __shared__ float lut[256];
    __shared__ float s_sa;
    lut[threadIdx.x] = ref_decode(threadIdx.x);
    __syncthreads();
    if (threadIdx.x == 0) {             // the query's norm fold (src/engine.rs:580), strictly in element order
        float sa = 0.0f;
        for (uint32_t i = 0; i < p.dim; ++i) { const float a = lut[p.qbytes[i]]; sa = ref_fold(sa, a, a); }
        s_sa = sa;
    }
    __syncthreads();
    const float sa = s_sa;
    const int sum_cq = p.qh->sum_cq;
    const uint32_t stride = gridDim.x * blockDim.x;
    const uint32_t lane = threadIdx.x & 31;
    // warp-uniform trip count: the ballot below needs every lane
    for (uint32_t i0 = blockIdx.x * blockDim.x; i0 < p.n_cand; i0 += stride) {
        const uint32_t i = i0 + threadIdx.x;
        bool ok = false;
        if (i < p.n_cand) {
            const uint32_t row = p.cand[i].x;
            const ReplayOut ro = replay_row<true>(p.rows + (size_t)row * p.pitch, p.qbytes, p.q16, p.dim, sum_cq, lut);
            const float dist = ref_distance(sa, ro.sb, ro.dot);
            const int64_t id = __ldg(p.ids + row);
            ok = dist < p.m && !page_before(p.cut, dist, id);
            if (p.recs) {
                p.key_dist[i] = ok ? ord_f32(dist) : 0xFFFFFFFFu;
                p.key_id[i] = (u64)id ^ 0x8000000000000000ull;
                p.index[i] = i;
                pbx_hit h;
                h.image_id = id; h.dist = dist; h.dot = ro.idot; h.norm2 = ro.inorm; h.flags = 0;
                p.recs[i] = h;
            }
        }
        const unsigned mask = __ballot_sync(0xFFFFFFFFu, ok);
        if (lane == 0 && mask) atomicAdd(p.counters + kRangeHits, (uint32_t)__popc(mask));
    }
}

// Between the two sorts: the dist keys in the order of the image_id sort.
__global__ void range_permute_keys_kernel(const uint32_t* __restrict__ key_dist, const uint32_t* __restrict__ index, uint32_t n,
                                          uint32_t* __restrict__ out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = key_dist[index[i]];
}

// The first n records in sorted order.
__global__ void range_gather_kernel(const pbx_hit* __restrict__ recs, const uint32_t* __restrict__ index, uint32_t n,
                                    pbx_hit* __restrict__ out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = recs[index[i]];
}

// Stable radix sorts of (key, value) pairs over all key bits (range_sort.cu); tmp = NULL: *tmp_bytes = the storage needed.
cudaError_t range_sort_pairs(void* tmp, size_t& tmp_bytes, const u64* keys_in, u64* keys_out, const uint32_t* vals_in,
                             uint32_t* vals_out, uint32_t n, cudaStream_t s);
cudaError_t range_sort_pairs(void* tmp, size_t& tmp_bytes, const uint32_t* keys_in, uint32_t* keys_out, const uint32_t* vals_in,
                             uint32_t* vals_out, uint32_t n, cudaStream_t s);

// The merge of a sharded range search: one shard's prefix src[0, n) packed into recs[at, at + n), with its sort keys.
__global__ void range_hit_keys_kernel(const pbx_hit* __restrict__ src, uint32_t n, uint32_t at, pbx_hit* __restrict__ recs,
                                      uint32_t* __restrict__ key_dist, u64* __restrict__ key_id, uint32_t* __restrict__ index) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const pbx_hit h = src[i];
        recs[at + i] = h;
        key_dist[at + i] = ord_f32(h.dist);
        key_id[at + i] = (u64)h.image_id ^ 0x8000000000000000ull;
        index[at + i] = at + i;
    }
}

}  // namespace pbx
