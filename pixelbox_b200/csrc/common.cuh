// common.cuh -- shared device helpers for the similarity-search kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "pixelbox_b200 kernels are written for sm_100a (B200) only"
#endif

namespace pbx {

typedef unsigned long long u64;

constexpr int kScanThreads = 256;            // 8 warps per scan CTA
constexpr int kScanWarps = kScanThreads / 32;
constexpr int kRowsPerWarpIter = 32;         // every warp iteration yields one row result per lane
constexpr int kItersPerTile = 4;             // generic kernel: warp iterations between two CTA-wide barriers
constexpr int kItersPerChunk = 4;            // fast kernel: warp iterations per claimed chunk
constexpr int kChunkRows = kRowsPerWarpIter * kItersPerChunk;              // 128 rows per warp claim
constexpr int kTileRows = kScanWarps * kRowsPerWarpIter * kItersPerTile;   // 1024 rows: push headroom of a CTA
constexpr int kFinalThreads = 1024;
constexpr int kMergeChunk = 4 * kFinalThreads;
constexpr uint32_t kMaxScanGrid = 2048;
constexpr uint32_t kHistBins = 4096;         // global histogram of candidate keys over kappa in [-1, 1]: 16 KB, one warp scans it in ~3 us
constexpr int kSeedThreads = 256;            // seed kernel: one sampled row per thread
constexpr uint32_t kMaxKeep = 3072;          // candidates per query the finalize kernel's shared memory is laid out for

// plateau value of the reference distance: 1/1e-6f - 1 evaluated in f32 (src/engine.rs:587)
#define PBX_PLATEAU_DIST 999999.0f

// ---- programmatic dependent launch (PDL) --------------------------------------------------------
// pdl_trigger(): lets the next kernel of the stream (launched with the programmatic-serialization attribute)
// start its independent prologue while this grid is still running.  pdl_wait(): blocks until every grid this
// one depends on has completed and its memory is visible.  Both are no-ops for a plain launch.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- integer dot products --------------------------------------------------------------
// dp2a: a holds two s16, b four u8.  lo: a.lo*b.byte0 + a.hi*b.byte1; hi: a.lo*b.byte2 + a.hi*b.byte3.
// SASS: IDP.2A.LO.S16.U8 / IDP.2A.HI.S16.U8.
__device__ __forceinline__ int dp2a_lo(int a, unsigned b, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi(int a, unsigned b, int c) {
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ unsigned dp4a_uu(unsigned a, unsigned b, unsigned c) {
    unsigned d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// streaming 16-byte load: read-only path, do not allocate in L1 (every corpus byte is used once per query)
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// ---- order-preserving float <-> uint ------------------------------------------------------
__device__ __host__ __forceinline__ uint32_t ord_f32(float f) {
#ifdef __CUDA_ARCH__
    uint32_t b = __float_as_uint(f);
#else
    union { float f; uint32_t u; } x; x.f = f; uint32_t b = x.u;
#endif
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __host__ __forceinline__ float unord_f32(uint32_t o) {
    uint32_t b = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    union { float f; uint32_t u; } x; x.u = b; return x.f;
#endif
}

// ---- the reference's f32 arithmetic, operation for operation (src/engine.rs:572-588) ------
// Every op is an explicit round-to-nearest intrinsic so nvcc can neither contract a*b+c into an
// FMA nor reassociate; Rust guarantees the same on the reference side.
__device__ __forceinline__ float ref_decode(uint32_t v) {   // ((*v as f32 / 255.0) * 2.0) - 1.0   :576
    return __fadd_rn(__fmul_rn(__fdiv_rn((float)v, 255.0f), 2.0f), -1.0f);
}
__device__ __forceinline__ float ref_fold(float init, float x, float y) {  // init + x*y            :580, :585
    return __fadd_rn(init, __fmul_rn(x, y));
}
__device__ __forceinline__ float ref_distance(float sa, float sb, float dot) {
    float magnitude = __fmul_rn(__fsqrt_rn(sa), __fsqrt_rn(sb));            // :581
    if (magnitude < 1e-6f) return 0.0f;                                     // :582-584
    float cosine_similarity = __fdiv_rn(dot, magnitude);                    // :586
    float m = fmaxf(cosine_similarity, 1e-6f);                              // f32::max (NaN cannot occur here)
    return __fadd_rn(__fdiv_rn(1.0f, m), -1.0f);                            // :587
}

// exact integer centring c(v) = 2v - 255 (SURVEY.md 8a R1)
__device__ __host__ __forceinline__ int centre(uint32_t v) { return 2 * (int)v - 255; }

// monotone map of the ranking key to a histogram bin (bin width 2 / kHistBins in cosine).  t = fl(kappa + 1) is
// formed with an explicit rounding so that "bin(kappa) >= b" and "t >= b / (bins/2)" are the same test
// (the multiplication by a power of two is exact).
__device__ __forceinline__ float kappa_shift(float kappa) { return __fadd_rn(kappa, 1.0f); }
__device__ __forceinline__ uint32_t kappa_bin(float kappa) {
    int b = __float2int_rd(__fmul_rn(kappa_shift(kappa), (float)(kHistBins / 2)));
    return (uint32_t)min(max(b, 0), (int)kHistBins - 1);
}
__device__ __forceinline__ float bin_threshold(uint32_t b) {      // kappa_shift(kappa) >= this  <=>  kappa_bin(kappa) >= b
    return b == 0 ? -__int_as_float(0x7f800000) : (float)b * (2.0f / (float)kHistBins);
}

// One warp: the highest bin b* with at least `keep` histogram entries at or above it (0 if there are
// fewer than `keep` entries).  Counts only grow while the scan runs, so a stale read is still valid.
__device__ inline uint32_t hist_threshold_warp(const uint32_t* hist, uint32_t keep, int lane) {
    constexpr uint32_t PER = kHistBins / 32;                      // lane l covers bins [l*PER, (l+1)*PER)
    const uint4* hp = reinterpret_cast<const uint4*>(hist + (size_t)lane * PER);
    uint32_t mine = 0;
#pragma unroll
    for (uint32_t i = 0; i < PER / 4; ++i) { const uint4 v = __ldcg(hp + i); mine += v.x + v.y + v.z + v.w; }
    uint32_t incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t v = __shfl_down_sync(0xFFFFFFFFu, incl, off);
        if (lane + off < 32) incl += v;
    }
    const uint32_t above = incl - mine;
    const bool has = above < keep && above + mine >= keep;
    uint32_t b = 0;
    if (has) {
        uint32_t run = above;
        for (int i = (int)PER - 1; i >= 0; --i) {
            run += __ldcg(hist + (size_t)lane * PER + i);
            if (run >= keep) { b = (uint32_t)lane * PER + (uint32_t)i; break; }
        }
    }
    const unsigned m = __ballot_sync(0xFFFFFFFFu, has);
    return m ? __shfl_sync(0xFFFFFFFFu, b, __ffs(m) - 1) : 0u;
}

// ---- filtered searches: one bit per row (mark_ids_kernel, filter.cuh); NULL = every row is allowed -----------------
__device__ __forceinline__ bool row_allowed(const uint32_t* allow, uint32_t row) {
    return allow == nullptr || ((__ldg(allow + (row >> 5)) >> (row & 31u)) & 1u) != 0u;
}

// ---- paged searches: the rows after a (dist, image_id) cursor (page.cuh derives one PageCut per query) -------------
// A row with kappa > kappa_hi sorts strictly before the cursor (DESIGN.md section 5): it is never pushed, sampled or
// replayed.  A row at or below the cut may still sort at or before the cursor; the replay decides (page_before).
struct PageCut {
    int64_t id0;                // cursor image_id
    float d0;                   // cursor dist
    float kappa_hi;             // +inf: no row is above the cut; -inf: every row is (the page is empty)
    uint32_t above;             // allowed rows the fast pass skipped for kappa > kappa_hi (an undercount is safe)
    uint32_t pad;
};
__device__ __forceinline__ float page_kappa_hi(const PageCut* cut) { return cut ? cut->kappa_hi : __int_as_float(0x7f800000); }
// (dist, id) <= (d0, id0): the row sorts at or before the cursor and is not on the page
__device__ __forceinline__ bool page_before(const PageCut* cut, float dist, int64_t id) {
    return cut != nullptr && (dist < cut->d0 || (dist == cut->d0 && id <= cut->id0));
}

// ---- candidate keys ----------------------------------------------------------------------
// fast pass: 64-bit key, larger is better: (ord(kappa) << 32) | ~row  (higher cosine first, then lower row)
__device__ __forceinline__ u64 make_key64(float kappa, uint32_t row) {
    return ((u64)ord_f32(kappa) << 32) | (u64)(0xFFFFFFFFu - row);
}
__device__ __forceinline__ uint32_t key64_row(u64 k) { return 0xFFFFFFFFu - (uint32_t)(k & 0xFFFFFFFFull); }
__device__ __forceinline__ float key64_kappa(u64 k) { return unord_f32((uint32_t)(k >> 32)); }

// exact pass: larger is better: (~ord(dist), ~biased id); the row rides along uncompared.
struct KeyX {
    uint32_t nd;    // ~ord_f32(dist): smaller distance -> larger
    uint32_t row;
    u64 nid;        // ~(id ^ sign): smaller image_id -> larger
};
__device__ __forceinline__ bool keyx_gt(const KeyX& a, const KeyX& b) {
    if (a.nd != b.nd) return a.nd > b.nd;
    if (a.nid != b.nid) return a.nid > b.nid;
    return a.row < b.row;
}
__device__ __forceinline__ KeyX make_keyx(float dist, int64_t id, uint32_t row) {
    KeyX k;
    k.nd = ~ord_f32(dist);
    k.row = row;
    k.nid = ~((u64)id ^ 0x8000000000000000ull);
    return k;
}
__device__ __forceinline__ int64_t keyx_id(const KeyX& k) { return (int64_t)((~k.nid) ^ 0x8000000000000000ull); }
__device__ __forceinline__ float keyx_dist(const KeyX& k) { return unord_f32(~k.nd); }

template <typename K> struct KeyOps;
template <> struct KeyOps<u64> {
    __device__ static __forceinline__ bool gt(const u64& a, const u64& b) { return a > b; }
    __device__ static __forceinline__ u64 lowest() { return 0ull; }
};
template <> struct KeyOps<KeyX> {
    __device__ static __forceinline__ bool gt(const KeyX& a, const KeyX& b) { return keyx_gt(a, b); }
    __device__ static __forceinline__ KeyX lowest() { KeyX k; k.nd = 0u; k.row = 0xFFFFFFFFu; k.nid = 0ull; return k; }
};

// ---- block-wide bitonic sort in shared memory, best (largest) first -------------------------
// n2 is a power of two; every thread of the block calls it.
template <typename K>
__device__ void block_sort_desc(K* buf, uint32_t n2) {
    for (uint32_t k = 2; k <= n2; k <<= 1) {
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < (n2 >> 1); t += blockDim.x) {
                uint32_t lo = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                uint32_t hi = lo | j;
                bool desc = (lo & k) == 0;
                K a = buf[lo], b = buf[hi];
                bool a_lt_b = KeyOps<K>::gt(b, a);
                if (a_lt_b == desc) { buf[lo] = b; buf[hi] = a; }
            }
            __syncthreads();
        }
    }
}

__device__ __host__ __forceinline__ uint32_t next_pow2(uint32_t v) {
    uint32_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

// Bounded candidate buffer of a CTA: pushes go through a warp-aggregated shared atomic; when the
// headroom for one more tile is gone the CTA sorts the buffer and keeps the best `keep`.
template <typename K>
struct TopBuf {
    K* buf;
    uint32_t* cnt;     // shared
    K* tau;            // shared: keep-th best so far (KeyOps::lowest() until `keep` entries exist)
    uint32_t cap;      // power of two
    uint32_t keep;

    __device__ __forceinline__ void push_warp(bool pass, const K& key) {
        unsigned m = __ballot_sync(0xFFFFFFFFu, pass);
        if (m == 0) return;
        unsigned lane = threadIdx.x & 31;
        int leader = __ffs(m) - 1;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(cnt, (uint32_t)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (pass) buf[base + __popc(m & ((1u << lane) - 1u))] = key;
    }
    // all threads; caller guarantees a barrier before (pushes complete).  Ends with a barrier.
    // Full sort, best first, cut to `keep`: used where the order matters (final lists); O(n log^2 n) barriers-heavy.
    __device__ void compact() {
        uint32_t c = *cnt;
        uint32_t n2 = next_pow2(c < 2 ? 2 : c);
        for (uint32_t i = c + threadIdx.x; i < n2; i += blockDim.x) buf[i] = KeyOps<K>::lowest();
        __syncthreads();
        block_sort_desc<K>(buf, n2);
        if (threadIdx.x == 0) {
            if (c >= keep) { *cnt = keep; *tau = buf[keep - 1]; }
        }
        __syncthreads();
    }
    // all threads; barrier before; ends with a barrier.  Keeps the entries for which pred holds, in place and
    // unordered: survivors of each block of blockDim entries are written below the region already read.
    template <typename Pred>
    __device__ void filter_inplace(Pred pred) {
        const uint32_t c0 = *cnt;
        __syncthreads();
        if (threadIdx.x == 0) *cnt = 0;
        for (uint32_t base = 0; base < c0; base += blockDim.x) {
            const uint32_t i = base + threadIdx.x;
            K e = KeyOps<K>::lowest();
            bool k = false;
            if (i < c0) { e = buf[i]; k = pred(e); }
            __syncthreads();
            push_warp(k, e);
        }
        __syncthreads();
    }
};

// Scratch of block_select_top.
struct SelectScratch {
    uint32_t hist[256];
    u64 prefix, mask;
    uint32_t need, stop;
};

// All threads; barrier before; ends with a barrier.  Cuts a buffer of unique u64 keys back to its `keep` largest
// (unordered) with an MSB-first radix select (8 bits per pass, stops as soon as a whole bucket is kept) and an
// in-place partition; *tau becomes the selection threshold (every kept key is >= it, no other key can equal it).
// Requires *cnt >= keep.  ~40 barriers instead of the ~80 steps x 8 pairs of a 4096-entry bitonic sort.
__device__ inline void block_select_top(TopBuf<u64>& tb, SelectScratch* sc) {
    const uint32_t c = *tb.cnt;
    if (threadIdx.x == 0) { sc->prefix = 0; sc->mask = 0; sc->need = tb.keep; sc->stop = 0; }
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) sc->hist[i] = 0;
        __syncthreads();
        const u64 prefix = sc->prefix, mask = sc->mask;
        for (uint32_t i = threadIdx.x; i < c; i += blockDim.x) {
            const u64 e = tb.buf[i];
            if ((e & mask) == prefix) atomicAdd(&sc->hist[(uint32_t)(e >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 32) {
            const uint32_t lane = threadIdx.x;
            uint32_t h[8], mine = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) { h[i] = sc->hist[lane * 8 + i]; mine += h[i]; }
            uint32_t incl = mine;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t v = __shfl_down_sync(0xFFFFFFFFu, incl, off);
                if (lane + off < 32) incl += v;
            }
            const uint32_t above = incl - mine, need = sc->need;
            __syncwarp();                                        // every lane has read `need` before the crossing lane rewrites it
            if (above < need && above + mine >= need) {          // exactly one lane
                uint32_t greater = above;
#pragma unroll
                for (int i = 7; i >= 0; --i) {
                    if (greater + h[i] >= need) {
                        sc->prefix = prefix | ((u64)(lane * 8 + i) << shift);
                        sc->mask = mask | (0xFFull << shift);
                        sc->need = need - greater;
                        if (h[i] == need - greater) sc->stop = 1;  // the whole bucket is kept: its lower edge is the threshold
                        break;
                    }
                    greater += h[i];
                }
            }
        }
        __syncthreads();
        if (sc->stop) break;
    }
    const u64 T = sc->prefix;
    tb.filter_inplace([T](const u64& e) { return e >= T; });
    if (threadIdx.x == 0) *tb.tau = T;
    __syncthreads();
}

}  // namespace pbx
