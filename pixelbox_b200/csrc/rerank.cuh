// rerank.cuh -- the tail of a fast-pass search, one CTA:
//   1. merge: the best `keep` keys of the union of the per-CTA candidate lists.  The scan CTAs add
//      their final lists to a global histogram over kappa; a suffix scan of it gives the bin b*
//      at which `keep` candidates are reached, every list contributes its (sorted) prefix with
//      bin >= b*, and the few hundred survivors are ordered by rank counting -- no barriers in the
//      sort, no passes over the 75k list entries.  Pathologically tied corpora (one bin holding
//      more than the buffer) fall back to threshold rounds over the rank-major lists.
//   2. kernel C: bit-exact f32 replay of the reference distance (src/engine.rs:572-588) for every
//      candidate: rows are staged in shared memory by all threads (one DRAM round trip), then one
//      thread per candidate folds its row strictly in element order.
//   3. ORDER BY dist ASC with ties by image_id, WHERE dist < max_dist, LIMIT k
//      (src/engine.rs:379-381), and the certificate that decides whether the exact pass runs.
#pragma once
#include "scan.cuh"
#include "../../include/pixelbox_b200.h"

namespace pbx {

struct FinalizeExactParams {
    const KeyX* cand;           // [k][grid] rank-major
    const uint32_t* cand_cnt;
    uint32_t grid;
    uint32_t k;
    uint32_t cap;               // power of two >= k + kMergeChunk
    uint32_t dim;
    uint32_t pitch;
    const uint8_t* rows;
    const uint8_t* qbytes;
    pbx_hit* hits;
    uint32_t* count;
    const SearchStatus* status;
    uint32_t* tile_counter;
    unsigned long long* exact_passes;
    uint32_t* done_flag;        // host-mapped word (or NULL): receives done_seq after the hits, with a system-scope fence between
    uint32_t done_seq;
};
__global__ void finalize_exact_kernel(const FinalizeExactParams p);     // finalize.cuh

// The exact (tie-resolving) pass is launched from the device, by the finalize kernel, only when the
// certificate fails: two tail launches (CUDA dynamic parallelism) that run after the finalize grid and
// before anything else in the stream.  A certified query -- the normal case -- pays nothing for it.
struct ExactLaunch {
    ScanParams scan;
    FinalizeExactParams fin;
    uint32_t grid, scan_smem, fin_smem, pad;
};

struct FinalizeParams {
    ExactLaunch x;
    const u64* cand;            // [keep][grid] rank-major, each CTA list sorted best first
    const uint32_t* cand_cnt;   // [grid]
    uint32_t* hist;             // [kHistBins] counts of the final list entries per kappa bin (zeroed here)
    uint32_t grid;              // scan CTAs
    uint32_t keep;              // k + slack
    uint32_t cap;               // key buffer capacity: power of two >= keep + chunk
    uint32_t chunk;             // fallback merge: elements per round, a multiple of kFinalThreads
    uint32_t k;
    uint32_t n;                 // rows searched
    const u64* n_allowed;       // filtered search: the number of allowed rows among them (device word), NULL = n
    const PageCut* cut;         // paged search: the cut and cursor of this query (batched: of query 0), NULL = first page
    uint32_t dim;
    uint32_t pitch;             // bytes
    uint32_t stage_rows;        // candidates per staging group (<= kFinalThreads: one thread per candidate)
    uint32_t slice16;           // 16-byte chunks of every candidate row staged per round
    // Split mode for large keep * pitch: phase 1 stops after the candidate selection and leaves the keys in x_keys /
    // x_meta, replay_kernel (many CTAs) replays the candidates into x_sbs / x_fdots / x_dots / x_norms, phase 2 picks
    // both up and orders, filters, writes the hits and the certificate.  phase 0: everything in this kernel.
    uint32_t phase;
    u64* x_keys;                // [keep]
    uint32_t* x_meta;           // {nc, kappa_k bits, kappa_last bits}
    float* x_sbs;               // [keep]
    float* x_fdots;             // [keep]
    int* x_dots;                // [keep]
    int* x_norms;               // [keep]
    uint32_t off_sorted;        // byte offsets into dynamic shared memory
    uint32_t off_ent, off_dots, off_q, off_stage;
    const uint8_t* rows;
    const int64_t* ids;
    const uint8_t* qbytes;      // this query, padded
    const int16_t* q16;         // this query, centred, padded
    QueryHeader* qh;            // sa is filled in here
    double max_dist;
    float margin;               // certificate margin on kappa (DESIGN.md section 5)
    pbx_hit* hits;              // [k] this query
    uint32_t* count;            // this query
    SearchStatus* status;       // this query
    uint32_t* tile_counter;     // reset for the next scan
    // Zero-copy completion (pbx_search_hits, one query): hits / count point into host-mapped memory and the host polls this
    // word instead of waiting for a copy and a stream synchronisation.  Written by whichever kernel produces the final
    // answer: this one, or finalize_exact_kernel when the exact pass runs.  NULL: not used.
    uint32_t* done_flag;
    uint32_t done_seq;
    // batched path (finalize_kernel<true>, one CTA per query; the per-query pointers above are those of query 0)
    const u64* bcand;           // [nq][kBatchCapacity] candidate keys (kappa' = dot_i * inv_norm_r, row)
    const uint32_t* bcnt;       // [nq]
    const uint32_t* boverflow;  // [nq] the candidate buffer overflowed: the exact pass must answer this query
    uint32_t* bticket;          // [2] zero on entry and on exit: ticket of the finished CTAs, count of queries needing the exact pass
    uint32_t bcap;              // entries per query in bcand
    uint32_t nq;
};

struct RerankEntry {            // sort record of kernel C: (ord(dist), image_id) ascending
    uint32_t od;
    uint32_t slot;
    int64_t id;
};
__device__ __forceinline__ bool rerank_before(const RerankEntry& a, const RerankEntry& b) {
    if (a.od != b.od) return a.od < b.od;
    if (a.id != b.id) return a.id < b.id;
    return a.slot < b.slot;
}
__device__ inline void block_sort_rerank(RerankEntry* e, uint32_t n2) {
    for (uint32_t k = 2; k <= n2; k <<= 1)
        for (uint32_t j = k >> 1; j > 0; j >>= 1) {
            for (uint32_t t = threadIdx.x; t < (n2 >> 1); t += blockDim.x) {
                uint32_t lo = ((t & ~(j - 1)) << 1) | (t & (j - 1)), hi = lo | j;
                bool asc = (lo & k) == 0;
                RerankEntry a = e[lo], b = e[hi];
                if (rerank_before(b, a) == asc) { e[lo] = b; e[hi] = a; }
            }
            __syncthreads();
        }
}

// Fallback merge: threshold rounds over the rank-major lists (strongest entries of every list first).
__device__ inline void merge_rounds(const FinalizeParams& p, TopBuf<u64>& tb, const uint32_t* s_listcnt, uint32_t maxcnt,
                                    uint32_t* s_pushed) {
    const uint32_t total = maxcnt * p.grid;
    for (uint32_t base = 0; base < total; base += p.chunk) {
        if (*tb.cnt + p.chunk > p.cap) tb.compact();        // uniform (read after a barrier)
        const u64 tau = *tb.tau;
        __syncthreads();
        if (threadIdx.x == 0) *s_pushed = 0;
        __syncthreads();
        bool any = false;
        for (uint32_t x = 0; x < p.chunk / kFinalThreads; ++x) {
            const uint32_t e = base + x * kFinalThreads + threadIdx.x;
            bool pass = false;
            u64 key = 0;
            if (e < total) {
                const uint32_t rank = e / p.grid, b = e - rank * p.grid;
                if (rank < s_listcnt[b]) { key = p.cand[e]; pass = key > tau; }
            }
            tb.push_warp(pass, key);
            any |= pass;
        }
        if (any) *s_pushed = 1;
        __syncthreads();
        // lists are sorted: a round that spans a complete rank and pushed nothing ends the merge
        if (*s_pushed == 0 && p.chunk >= 2 * p.grid) break;
    }
    __syncthreads();
    tb.compact();
}

// 16 staged row bytes against 16 decoded query floats, strictly in element order
__device__ __forceinline__ void fold16(const uint4& v, const float* qa, const float* lut, float& s, float& d) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 a = *reinterpret_cast<const float4*>(qa + 4 * i);
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const float fb = lut[(w[i] >> (8 * b)) & 255u];
            s = ref_fold(s, fb, fb);
            d = ref_fold(d, av[b], fb);
        }
    }
}

// One 16-byte chunk (index ch within the row) of a candidate against the query: the two f32 folds of the reference in
// element order, and the exact integer sums beside them.
__device__ __forceinline__ void replay_chunk(const uint4& v, uint32_t ch, uint32_t full, uint32_t dim, const float* s_qa,
                                             const int16_t* s_q16, const float* s_lut, float& s, float& d, int& acc, unsigned& s1,
                                             unsigned& s2) {
    if (ch < full) {
        fold16(v, s_qa + 16 * ch, s_lut, s, d);
    } else {                                            // ragged tail: dim is not a multiple of 16
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
        for (uint32_t i = 16 * ch; i < dim; ++i) {
            const uint32_t o = i - 16 * ch;
            const float fb = s_lut[(w[o >> 2] >> (8 * (o & 3))) & 255u];
            s = ref_fold(s, fb, fb);
            d = ref_fold(d, s_qa[i], fb);
        }
    }
    const int4 qa4 = *reinterpret_cast<const int4*>(s_q16 + 16 * ch), qb4 = *reinterpret_cast<const int4*>(s_q16 + 16 * ch + 8);
    const int qq[8] = {qa4.x, qa4.y, qa4.z, qa4.w, qb4.x, qb4.y, qb4.z, qb4.w};
    acc = dot16(v, qq, acc);
    s1 = dp4a_uu(v.x, 0x01010101u, s1); s1 = dp4a_uu(v.y, 0x01010101u, s1);
    s1 = dp4a_uu(v.z, 0x01010101u, s1); s1 = dp4a_uu(v.w, 0x01010101u, s1);
    s2 = dp4a_uu(v.x, v.x, s2); s2 = dp4a_uu(v.y, v.y, s2);
    s2 = dp4a_uu(v.z, v.z, s2); s2 = dp4a_uu(v.w, v.w, s2);
}

// ---- the replay of the candidates on many SMs (split finalize) ----------------------------------------------------------
// One CTA per 32 candidates: 256 threads stage slices of the 32 rows, the lanes of warp 0 each fold one candidate.  The
// folds are strictly sequential per candidate, so what this buys is all candidates at once at one SM's latency each,
// instead of one SM's instruction throughput for keep * dim elements.
constexpr uint32_t kReplayRows = 32, kReplayThreads = 256, kReplaySlice16 = 31;
struct ReplayParams {
    const u64* keys;
    const uint32_t* meta;
    const uint8_t* rows;
    const uint8_t* qbytes;
    const int16_t* q16;
    const QueryHeader* qh;
    uint32_t dim, pitch;
    float* sbs;
    float* fdots;
    int* dots;
    int* norms;
};

__global__ void __launch_bounds__(kReplayThreads)
replay_kernel(const ReplayParams p) {
    extern __shared__ __align__(16) unsigned char rsm[];
    float* s_qa = reinterpret_cast<float*>(rsm);                                       // [pitch]
    int16_t* s_q16 = reinterpret_cast<int16_t*>(rsm + 4 * (size_t)p.pitch);            // [pitch]
    unsigned char* stage = rsm + 6 * (size_t)p.pitch;                                   // [32][33 * 16]
    __shared__ float s_lut[256];
    __shared__ uint32_t s_rows[kReplayRows];
    const uint32_t tid = threadIdx.x;
    const uint32_t nc = p.meta[0];
    const uint32_t c0 = blockIdx.x * kReplayRows;
    if (c0 >= nc) return;
    const uint32_t cb = min(kReplayRows, nc - c0);
    s_lut[tid] = ref_decode(tid);
    if (tid < cb) s_rows[tid] = key64_row(p.keys[c0 + tid]);
    for (uint32_t i = tid; i < p.pitch / 8; i += blockDim.x)
        reinterpret_cast<uint4*>(s_q16)[i] = __ldg(reinterpret_cast<const uint4*>(p.q16) + i);
    __syncthreads();
    for (uint32_t i = tid; i < p.pitch; i += blockDim.x) s_qa[i] = s_lut[p.qbytes[i]];
    __syncthreads();
    const uint32_t pitch16 = p.pitch / 16, full = p.dim >> 4;
    constexpr uint32_t srow = (kReplaySlice16 + 2) * 16;        // 33 x 16 bytes: an odd number of 16-byte units
    float s = 0.0f, d = 0.0f;
    int acc = 0;
    unsigned s1 = 0, s2 = 0;
    for (uint32_t ch0 = 0; ch0 < pitch16; ch0 += kReplaySlice16) {
        const uint32_t w16 = min(kReplaySlice16, pitch16 - ch0);
        const uint32_t total16 = cb * w16;
        for (uint32_t e0 = tid; e0 < total16; e0 += 4 * blockDim.x) {
            uint4 v[4];
#pragma unroll
            for (uint32_t u = 0; u < 4; ++u) {
                const uint32_t e = e0 + u * blockDim.x;
                if (e < total16) {
                    const uint32_t ci = e / w16, ch = e - ci * w16;
                    v[u] = __ldg(reinterpret_cast<const uint4*>(p.rows + (size_t)s_rows[ci] * p.pitch) + ch0 + ch);
                }
            }
#pragma unroll
            for (uint32_t u = 0; u < 4; ++u) {
                const uint32_t e = e0 + u * blockDim.x;
                if (e < total16) {
                    const uint32_t ci = e / w16, ch = e - ci * w16;
                    *reinterpret_cast<uint4*>(stage + (size_t)ci * srow + 16 * ch) = v[u];
                }
            }
        }
        __syncthreads();
        if (tid < cb) {
            const unsigned char* r = stage + (size_t)tid * srow;
            for (uint32_t cl = 0; cl < w16; ++cl)
                replay_chunk(*reinterpret_cast<const uint4*>(r + 16 * cl), ch0 + cl, full, p.dim, s_qa, s_q16, s_lut, s, d, acc, s1, s2);
        }
        __syncthreads();
    }
    if (tid < cb) {
        p.sbs[c0 + tid] = s;
        p.fdots[c0 + tid] = d;
        p.dots[c0 + tid] = 2 * acc - 255 * p.qh->sum_cq;
        p.norms[c0 + tid] = (int)(4u * s2 - 1020u * s1 + 65025u * p.dim);
    }
}

// out_count marker of a query whose exact pass could not be launched from the device (the pending-launch pool was
// exhausted): the fast-pass hits in the output are NOT certified.  The host-buffer API re-runs the exact pass from the
// host when it sees it; callers of the device-resident API must treat it as PBX_E_INTERNAL for that query.
// (PBX_COUNT_EXACT_LAUNCH_FAILED, include/pixelbox_b200.h)

#ifdef PBX_USE_CDP
// Returns false if either tail launch was refused (cudaGetLastError is part of the device runtime).
__device__ inline bool launch_exact_tail(const ExactLaunch& x) {
#define PBX_X_CASE(LL, CC) \
    case LL * CC: scan_kernel<LL, CC, true><<<x.grid, kScanThreads, x.scan_smem, cudaStreamTailLaunch>>>(x.scan); break;
    switch (x.scan.pitch16) {
        PBX_X_CASE(1, 1) PBX_X_CASE(2, 1) PBX_X_CASE(4, 1) PBX_X_CASE(8, 1) PBX_X_CASE(16, 1) PBX_X_CASE(32, 1)
        PBX_X_CASE(32, 2) PBX_X_CASE(32, 4)
#define PBX_X_CASE_M(LL, CC, MM) \
    case (LL) * (CC): scan_kernel<LL, CC, true, MM><<<x.grid, kScanThreads, x.scan_smem, cudaStreamTailLaunch>>>(x.scan); break;
        PBX_EXTRA_SHAPES(PBX_X_CASE_M)
#undef PBX_X_CASE_M
        default:
            scan_generic_kernel<true><<<x.grid, kScanThreads, x.scan_smem + x.scan.pitch16 * 32, cudaStreamTailLaunch>>>(x.scan);
            break;
    }
#undef PBX_X_CASE
    if (cudaGetLastError() != cudaSuccess) return false;
    finalize_exact_kernel<<<1, kFinalThreads, x.fin_smem, cudaStreamTailLaunch>>>(x.fin);
    return cudaGetLastError() == cudaSuccess;
}
#endif

#ifdef PBX_EXP_PROFILE
__device__ long long g_fin_prof[16];     // experiment builds only: clock64 stamps of the finalize phases
#define PBX_FIN_STAMP(i) do { if (threadIdx.x == 0) g_fin_prof[i] = clock64(); } while (0)
#else
#define PBX_FIN_STAMP(i) do { } while (0)
#endif

// Orders m unique keys best-first from buf into sorted: rank counting when small (no barriers), bitonic otherwise.
// All threads; barrier before; ends with a barrier.  buf may be clobbered.
__device__ inline void block_order_keys(u64* buf, u64* sorted, uint32_t m) {
    const uint32_t tid = threadIdx.x;
    if (m <= kFinalThreads) {
        // TPE threads share one element: each counts a strided part of the buffer, shuffles add up
        const uint32_t tpe = min(32u, (uint32_t)kFinalThreads / next_pow2(m < 2 ? 2 : m));
        const uint32_t e = tid / tpe, sub = tid - e * tpe;
        const u64 me = e < m ? buf[e] : 0ull;
        uint32_t rank = 0;
        if (e < m) {                                       // idle groups only take part in the shuffles
#pragma unroll 4
            for (uint32_t j = sub; j < m; j += tpe) rank += (buf[j] > me) ? 1u : 0u;
        }
        for (uint32_t off = tpe >> 1; off; off >>= 1) rank += __shfl_xor_sync(0xFFFFFFFFu, rank, off);
        if (e < m && sub == 0) sorted[rank] = me;
        __syncthreads();
    } else if (m <= 2 * kFinalThreads) {
        for (uint32_t t = tid; t < m; t += blockDim.x) {
            const u64 me = buf[t];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < m; ++j) rank += (buf[j] > me) ? 1u : 0u;
            sorted[rank] = me;
        }
        __syncthreads();
    } else {
        const uint32_t m2 = next_pow2(m);
        for (uint32_t i = m + tid; i < m2; i += blockDim.x) buf[i] = 0ull;
        __syncthreads();
        block_sort_desc<u64>(buf, m2);
        for (uint32_t i = tid; i < m; i += blockDim.x) sorted[i] = buf[i];
        __syncthreads();
    }
}

// Smallest key of a[0..n) (n >= 1), all threads; barrier before; ends with a barrier.  Result in *s_out (shared).
__device__ inline void block_min_key(const u64* a, uint32_t n, u64* s_out, u64* s_scratch /* [32] shared */) {
    u64 m = ~0ull;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) m = a[i] < m ? a[i] : m;
    for (int off = 16; off; off >>= 1) {
        const u64 o = __shfl_xor_sync(0xFFFFFFFFu, m, off);
        m = o < m ? o : m;
    }
    if ((threadIdx.x & 31) == 0) s_scratch[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        u64 r = ~0ull;
        for (uint32_t w = 0; w < (blockDim.x + 31) / 32; ++w) r = s_scratch[w] < r ? s_scratch[w] : r;
        *s_out = r;
    }
    __syncthreads();
}

// From m unique keys in buf to the candidate set: the best min(m, keep) keys in sorted[0..nc) plus the kappa of
// the k-th and of the last of them (what the certificate needs).  Small sets are fully ordered by rank counting;
// large ones (large k) only go through two radix selects and two min-reductions -- the order by kappa is never
// needed downstream.  All threads; barrier before; ends with a barrier.  buf is clobbered.
__device__ inline uint32_t block_candidates(u64* buf, u64* sorted, uint32_t m, uint32_t keep, uint32_t k, uint32_t cap,
                                            uint32_t* s_cnt, u64* s_tau, SelectScratch* s_sel, u64* s_scratch,
                                            float* s_kappa_k, float* s_kappa_last) {
    if (m <= kFinalThreads) {
        block_order_keys(buf, sorted, m);
        const uint32_t nc = m < keep ? m : keep;
        if (threadIdx.x == 0) {
            *s_kappa_k = (nc >= k && k > 0) ? key64_kappa(sorted[k - 1]) : 0.0f;
            *s_kappa_last = nc > 0 ? key64_kappa(sorted[nc - 1]) : 0.0f;
        }
        __syncthreads();
        return nc;
    }
    TopBuf<u64> tb{buf, s_cnt, s_tau, cap, keep};
    if (threadIdx.x == 0) *s_cnt = m;
    __syncthreads();
    if (m > keep) block_select_top(tb, s_sel);
    const uint32_t nc = *s_cnt;
    for (uint32_t i = threadIdx.x; i < nc; i += blockDim.x) sorted[i] = buf[i];
    __syncthreads();
    __shared__ u64 s_min;
    block_min_key(sorted, nc, &s_min, s_scratch);
    if (threadIdx.x == 0) *s_kappa_last = key64_kappa(s_min);
    if (nc > k && k > 0) {
        TopBuf<u64> tk{buf, s_cnt, s_tau, cap, k};
        block_select_top(tk, s_sel);                       // buf is scratch from here on
        block_min_key(buf, k, &s_min, s_scratch);
        if (threadIdx.x == 0) *s_kappa_k = key64_kappa(s_min);
    } else if (threadIdx.x == 0) {
        *s_kappa_k = (nc == k && k > 0) ? key64_kappa(s_min) : 0.0f;
    }
    __syncthreads();
    return nc;
}

template <bool BATCH>
__global__ void __launch_bounds__(kFinalThreads, 1)
finalize_kernel(const FinalizeParams p) {
    PBX_FIN_STAMP(0);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64* buf = reinterpret_cast<u64*>(smem_raw);                                   // [cap]
    u64* sorted = reinterpret_cast<u64*>(smem_raw + p.off_sorted);                 // [cap]
    RerankEntry* ent = reinterpret_cast<RerankEntry*>(smem_raw + p.off_ent);       // [next_pow2(keep)]
    int* dots = reinterpret_cast<int*>(smem_raw + p.off_dots);                     // [keep]
    int* norms = dots + p.keep;
    float* dists = reinterpret_cast<float*>(norms + p.keep);
    float* sbs = dists + p.keep;
    float* fdots = sbs + p.keep;
    float* s_qa = reinterpret_cast<float*>(smem_raw + p.off_q);                    // [pitch] decoded query
    int16_t* s_q16 = reinterpret_cast<int16_t*>(smem_raw + p.off_q + 4 * p.pitch); // [pitch] centred query
    unsigned char* stage = smem_raw + p.off_stage;                                 // [stage_rows][slice16 * 16 + 16]

    __shared__ uint32_t s_cnt, s_pushed, s_maxcnt, s_nonplateau, s_bstar, s_mprime, s_total, s_odlo, s_odhi, s_excl, s_scnt;
    __shared__ u64 s_tau;
    __shared__ float s_lut[256];
    __shared__ float s_kappa_k, s_kappa_last, s_sa;
    __shared__ uint32_t s_listcnt[kMaxScanGrid];
    __shared__ uint32_t s_warp[32];
    __shared__ u64 s_scratch64[32];

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t q = BATCH ? blockIdx.x : 0u;
    const int16_t* q16_g = p.q16 + (size_t)q * p.pitch;
    const uint8_t* qbytes_g = p.qbytes + (size_t)q * p.pitch;
    QueryHeader* qh_g = p.qh + q;
    pbx_hit* hits_g = p.hits + (size_t)q * p.k;
    uint32_t* count_g = p.count + q;
    SearchStatus* status_g = p.status + q;
    const PageCut* cut_g = p.cut ? p.cut + q : nullptr;
    __shared__ SelectScratch s_sel;
    // No pdl_trigger() here: this grid may tail-launch the exact pass, which must run before anything else in
    // the stream; a next-query kernel that was already started early would wait for it while it waits for them.
    if (tid < 256) s_lut[tid] = ref_decode(tid);
    if (tid == 0) { s_cnt = 0; s_tau = 0ull; s_maxcnt = 0; s_nonplateau = 0; s_pushed = 0; s_bstar = 0; s_mprime = 0; s_odlo = 0xFFFFFFFFu; s_odhi = 0u; s_excl = 0; s_scnt = 0; }
    pdl_wait();                 // the scan is complete: lists, histogram and the query scratch are visible
    for (uint32_t i = tid; i < p.pitch / 8; i += blockDim.x)
        reinterpret_cast<uint4*>(s_q16)[i] = __ldg(reinterpret_cast<const uint4*>(q16_g) + i);
    __syncthreads();
    for (uint32_t i = tid; i < p.pitch; i += blockDim.x) s_qa[i] = s_lut[qbytes_g[i]];
    uint32_t nc;
    if (!BATCH && p.phase == 2) {
        // split mode, second half: the candidate keys come back from the first half
        nc = p.x_meta[0];
        for (uint32_t i = tid; i < nc; i += blockDim.x) sorted[i] = p.x_keys[i];
        if (tid == 0) { s_kappa_k = __uint_as_float(p.x_meta[1]); s_kappa_last = __uint_as_float(p.x_meta[2]); }
        __syncthreads();
    } else if constexpr (!BATCH) {
        for (uint32_t b = tid; b < p.grid; b += blockDim.x) {
            uint32_t c = p.cand_cnt[b];
            s_listcnt[b] = c;
            atomicMax(&s_maxcnt, c);
        }

        PBX_FIN_STAMP(1);
        // ---- 1a. histogram suffix scan: b* = highest bin with at least `keep` entries at or above it -------
        constexpr uint32_t BPT = kHistBins / kFinalThreads;            // bins per thread
        uint32_t h[BPT];
    #pragma unroll
        for (uint32_t i = 0; i < BPT; ++i) {
            h[i] = __ldcg(p.hist + (size_t)tid * BPT + i);
            p.hist[(size_t)tid * BPT + i] = 0;                         // ready for the next query
        }
        uint32_t mine = 0;
    #pragma unroll
        for (uint32_t i = 0; i < BPT; ++i) mine += h[i];
        // inclusive suffix sum over threads (thread t covers bins [t*BPT, (t+1)*BPT)): above = entries in higher threads
        uint32_t incl = mine;
    #pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            uint32_t v = __shfl_down_sync(0xFFFFFFFFu, incl, off);
            if (lane + off < 32) incl += v;
        }
        if (lane == 0) s_warp[warp] = incl;
        __syncthreads();
        uint32_t above = incl - mine;
        for (uint32_t w = warp + 1; w < kFinalThreads / 32; ++w) above += s_warp[w];
        if (tid == 0) { uint32_t t = 0; for (uint32_t w = 0; w < kFinalThreads / 32; ++w) t += s_warp[w]; s_total = t; }
        if (above < p.keep && above + mine >= p.keep) {                // the crossing bin is one of mine
            uint32_t run = above;
    #pragma unroll
            for (int i = BPT - 1; i >= 0; --i) {
                run += h[i];
                if (run >= p.keep) { s_bstar = tid * BPT + i; s_mprime = run; break; }
            }
        }
        __syncthreads();
        if (s_total < p.keep && tid == 0) { s_bstar = 0; s_mprime = s_total; }   // fewer entries than keep: take everything
        __syncthreads();

        PBX_FIN_STAMP(2);
        const uint32_t mprime = s_mprime, bstar = s_bstar;
        if (mprime <= p.cap) {
            // ---- 1b. gather the list prefixes with bin >= b* ---------------------------------------------
            for (uint32_t b = tid; b < p.grid; b += blockDim.x) {
                const uint32_t len = s_listcnt[b];
                for (uint32_t r0 = 0; r0 < len; r0 += 4) {
                    u64 key[4];
    #pragma unroll
                    for (uint32_t i = 0; i < 4; ++i) key[i] = (r0 + i < len) ? p.cand[(size_t)(r0 + i) * p.grid + b] : 0ull;
                    uint32_t take = 0;
    #pragma unroll
                    for (uint32_t i = 0; i < 4; ++i)
                        if (take == i && r0 + i < len && kappa_bin(key64_kappa(key[i])) >= bstar) take = i + 1;
                    if (take) {
                        const uint32_t at = atomicAdd(&s_cnt, take);
    #pragma unroll
                        for (uint32_t i = 0; i < 4; ++i) if (i < take) buf[at + i] = key[i];
                    }
                    if (take < 4) break;
                }
            }
            __syncthreads();
            PBX_FIN_STAMP(3);
            const uint32_t m = s_cnt;                                   // <= mprime
            // ---- 1c. candidate set + the two kappas of the certificate ------------------------------------
            nc = block_candidates(buf, sorted, m, p.keep, p.k, p.cap, &s_cnt, &s_tau, &s_sel, s_scratch64, &s_kappa_k, &s_kappa_last);
        } else {
            // ---- 1'. fallback: more ties in one bin than the buffer holds ----------------------------------
            TopBuf<u64> tb{buf, &s_cnt, &s_tau, p.cap, p.keep};
            merge_rounds(p, tb, s_listcnt, s_maxcnt, &s_pushed);
            nc = s_cnt < p.keep ? s_cnt : p.keep;
            for (uint32_t i = tid; i < nc; i += blockDim.x) sorted[i] = buf[i];
            __syncthreads();
            if (tid == 0) {                                   // merge_rounds leaves the buffer sorted best first
                s_kappa_k = (nc >= p.k && p.k > 0) ? key64_kappa(sorted[p.k - 1]) : 0.0f;
                s_kappa_last = nc > 0 ? key64_kappa(sorted[nc - 1]) : 0.0f;
            }
            __syncthreads();
        }
    } else {
        // ---- 1 (batched). this query's candidate buffer: kappa' -> kappa, cut to `keep`, order ---------------
        __syncthreads();
        const uint32_t c = min(min(p.bcnt[q], p.bcap), p.cap);       // p.cap: what this kernel's shared buffers hold
        const float inv_q = qh_g->inv_q;
        const u64* src = p.bcand + (size_t)q * p.bcap;
        for (uint32_t i = tid; i < c; i += blockDim.x) {
            const u64 e = src[i];
            buf[i] = make_key64(__fmul_rn(key64_kappa(e), inv_q), key64_row(e));
        }
        if (tid == 0) s_cnt = c;
        __syncthreads();
        if (c > p.keep) {
            TopBuf<u64> tb{buf, &s_cnt, &s_tau, p.cap, p.keep};
            block_select_top(tb, &s_sel);
        }
        const uint32_t m = s_cnt;
        nc = block_candidates(buf, sorted, m, p.keep, p.k, p.cap, &s_cnt, &s_tau, &s_sel, s_scratch64, &s_kappa_k, &s_kappa_last);
    }

    PBX_FIN_STAMP(4);
    if (!BATCH && p.phase == 1) {
        // split mode, first half: hand the candidate keys to replay_kernel and to the second half
        for (uint32_t i = tid; i < nc; i += blockDim.x) p.x_keys[i] = sorted[i];
        if (tid == 0) { p.x_meta[0] = nc; p.x_meta[1] = __float_as_uint(s_kappa_k); p.x_meta[2] = __float_as_uint(s_kappa_last); }
        return;
    }
    // ---- 2. kernel C ------------------------------------------------------------------------------------
    // The query's own norm fold (src/engine.rs:580): the products in parallel (same rounding), the strictly sequential
    // additions by one thread of the last warp, eight loads ahead of the 4-cycle add chain.  The squares live in `buf`,
    // which is dead between the candidate selection and the sort records; nobody else waits for this thread before the
    // first barrier of the staging loop.
    {
        float* sq = reinterpret_cast<float*>(buf);
        for (uint32_t i = tid; i < p.dim; i += blockDim.x) { const float a = s_qa[i]; sq[i] = __fmul_rn(a, a); }
        __syncthreads();
        if (tid == kFinalThreads - 1) {
            float sa = 0.0f;
            uint32_t i = 0;
            for (; i + 8 <= p.dim; i += 8) {
                const float4 x = *reinterpret_cast<const float4*>(sq + i), y = *reinterpret_cast<const float4*>(sq + i + 4);
                sa = __fadd_rn(sa, x.x); sa = __fadd_rn(sa, x.y); sa = __fadd_rn(sa, x.z); sa = __fadd_rn(sa, x.w);
                sa = __fadd_rn(sa, y.x); sa = __fadd_rn(sa, y.y); sa = __fadd_rn(sa, y.z); sa = __fadd_rn(sa, y.w);
            }
            for (; i < p.dim; ++i) sa = __fadd_rn(sa, sq[i]);
            s_sa = sa;
            qh_g->sa = sa;
        }
    }
    // Candidate rows are staged in shared memory in COLUMN SLICES: every thread owns one candidate (groups of up to
    // 1024) and carries its five partial sums in registers from slice to slice, so all candidates advance together
    // whatever the row length.  (Staging whole rows would serialise the strictly sequential f32 folds of a long row
    // over a handful of rows at a time: 8 rounds of 45 rows at dim 4096.)
    const uint32_t pitch16 = p.pitch / 16, slice16 = p.slice16;
    const uint32_t srow = ((slice16 + 1) | 1u) * 16;            // row stride: an odd number of 16-byte units (no bank conflicts)
    const uint32_t full = p.dim >> 4;
    const int sum_cq = qh_g->sum_cq;
    constexpr uint32_t kStageBatch = 6;
    if (!BATCH && p.phase == 2) {
        for (uint32_t i = tid; i < nc; i += blockDim.x) {
            sbs[i] = p.x_sbs[i]; fdots[i] = p.x_fdots[i]; dots[i] = p.x_dots[i]; norms[i] = p.x_norms[i];
        }
    } else
    for (uint32_t c0 = 0; c0 < nc; c0 += p.stage_rows) {
        const uint32_t cb = min(p.stage_rows, nc - c0);                // <= blockDim.x
        float s = 0.0f, d = 0.0f;
        int acc = 0;
        unsigned s1 = 0, s2 = 0;
        for (uint32_t ch0 = 0; ch0 < pitch16; ch0 += slice16) {
            const uint32_t w16 = min(slice16, pitch16 - ch0);
            // all threads: one 16-byte load per (candidate, chunk of the slice), kStageBatch of them in flight per thread
            // before the first store (a load -> store loop keeps ONE in flight: the candidates are random rows, every
            // load is a DRAM + TLB miss)
            const uint32_t total16 = cb * w16;
            for (uint32_t e0 = tid; e0 < total16; e0 += kStageBatch * blockDim.x) {
                uint4 v[kStageBatch];
#pragma unroll
                for (uint32_t u = 0; u < kStageBatch; ++u) {
                    const uint32_t e = e0 + u * blockDim.x;
                    if (e < total16) {
                        const uint32_t ci = e / w16, ch = e - ci * w16;
                        const uint32_t row = key64_row(sorted[c0 + ci]);
                        v[u] = __ldg(reinterpret_cast<const uint4*>(p.rows + (size_t)row * p.pitch) + ch0 + ch);
                    }
                }
#pragma unroll
                for (uint32_t u = 0; u < kStageBatch; ++u) {
                    const uint32_t e = e0 + u * blockDim.x;
                    if (e < total16) {
                        const uint32_t ci = e / w16, ch = e - ci * w16;
                        *reinterpret_cast<uint4*>(stage + (size_t)ci * srow + 16 * ch) = v[u];
                    }
                }
            }
            __syncthreads();
            PBX_FIN_STAMP(5);
            if (tid < cb) {
                const unsigned char* r = stage + (size_t)tid * srow;
                for (uint32_t cl = 0; cl < w16; ++cl)
                    replay_chunk(*reinterpret_cast<const uint4*>(r + 16 * cl), ch0 + cl, full, p.dim, s_qa, s_q16, s_lut, s, d, acc, s1, s2);
            }
            __syncthreads();
        }
        if (tid < cb) {
            sbs[c0 + tid] = s;
            fdots[c0 + tid] = d;
            dots[c0 + tid] = 2 * acc - 255 * sum_cq;
            norms[c0 + tid] = (int)(4u * s2 - 1020u * s1 + 65025u * p.dim);
        }
    }
    __syncthreads();
    PBX_FIN_STAMP(6);
    const float sa = s_sa;
    const uint32_t n2 = next_pow2(nc < 2 ? 2 : nc);
    uint32_t nonplateau = 0;
    // ent overlays buf/sorted: fetch the image ids (and the keys, for a paged search) through `sorted` first, write ent
    // after a barrier
    int64_t my_id[kMaxKeep / kFinalThreads];
    u64 my_key[kMaxKeep / kFinalThreads];
    uint32_t my_excl = 0;                                   // bit x: candidate tid + x * kFinalThreads sorts at or before the cursor
#pragma unroll
    for (uint32_t x = 0; x < kMaxKeep / kFinalThreads; ++x) {
        const uint32_t c = tid + x * kFinalThreads;
        my_key[x] = (c < nc) ? sorted[c] : 0ull;
        my_id[x] = (c < nc) ? p.ids[key64_row(my_key[x])] : INT64_MAX;
    }
    __syncthreads();
    uint32_t excl = 0;
#pragma unroll
    for (uint32_t x = 0; x < kMaxKeep / kFinalThreads; ++x) {
        const uint32_t c = tid + x * kFinalThreads;
        if (c < nc) {
            const float dist = ref_distance(sa, sbs[c], fdots[c]);
            RerankEntry e;
            e.slot = c;
            if (page_before(cut_g, dist, my_id[x])) {
                // Paged search: not on the page.  It is taken out of the ranking -- it sorts after every real row, never
                // passes, and is not a surviving candidate for the certificate -- rather than only marked: with its
                // real dist it would sort first.
                dists[c] = __int_as_float(0x7fffffff);         // NaN: never < max_dist
                e.od = 0xFFFFFFFFu;
                e.id = INT64_MAX;
                my_excl |= 1u << x;
                ++excl;
            } else {
                dists[c] = dist;
                e.od = ord_f32(dist);
                e.id = my_id[x];
                if (dist < PBX_PLATEAU_DIST) nonplateau++;
            }
            ent[c] = e;
        }
    }
    if (excl) atomicAdd(&s_excl, excl);
    for (uint32_t c = nc + tid; c < n2; c += blockDim.x) {
        RerankEntry e; e.od = 0xFFFFFFFFu; e.slot = 0xFFFFFFFFu; e.id = INT64_MAX;
        ent[c] = e;
    }
    if (nonplateau) atomicAdd(&s_nonplateau, nonplateau);
    if (tid == 0) s_cnt = 0;
    __syncthreads();

    PBX_FIN_STAMP(7);
    // ---- 3. ORDER BY dist ASC (ties by image_id), WHERE dist < ?, LIMIT k  (engine.rs:379-381) ---------
    // `pos` = position of candidate c in the final order; ascending order makes the passing rows a prefix
    uint32_t local = 0;
    if (nc <= kFinalThreads) {
        // rank counting, TPE threads per candidate, no barriers
        const uint32_t tpe = min(32u, (uint32_t)kFinalThreads / next_pow2(nc < 2 ? 2 : nc));
        const uint32_t c = tid / tpe, sub = tid - c * tpe;
        RerankEntry me; me.od = 0; me.slot = 0; me.id = 0;
        if (c < nc) me = ent[c];
        uint32_t pos = 0;
        if (c < nc) {
#pragma unroll 4
            for (uint32_t j = sub; j < nc; j += tpe) pos += rerank_before(ent[j], me) ? 1u : 0u;
        }
        for (uint32_t off = tpe >> 1; off; off >>= 1) pos += __shfl_xor_sync(0xFFFFFFFFu, pos, off);
        if (c < nc && sub == 0) {
            const float dist = dists[c];
            const bool ok = (double)dist < p.max_dist;
            if (ok) local = 1;
            if (pos < p.k) {
                pbx_hit hh;
                if (ok) { hh.image_id = me.id; hh.dist = dist; hh.dot = dots[c]; hh.norm2 = norms[c]; hh.flags = 0; }
                else { hh.image_id = INT64_MAX; hh.dist = __int_as_float(0x7f800000); hh.dot = 0; hh.norm2 = 0; hh.flags = 0; }
                hits_g[pos] = hh;
            }
        }
    } else if ((size_t)nc * sizeof(RerankEntry) <= p.off_sorted) {
        // Large k: up to 1024 order-preserving buckets over [min od, max od] (a shift of od - min), entries scattered bucket by bucket, then rank
        // counting inside each bucket only (a handful of entries unless many distances tie exactly, e.g. on the
        // plateau: then it degrades to plain rank counting, still correct).  ~10x cheaper than a bitonic sort of
        // 16-byte records.  `sorted` is free by now (the ids were fetched through it above) and holds the scatter.
        RerankEntry* ent2 = reinterpret_cast<RerankEntry*>(sorted);
        uint32_t* s_base = s_listcnt;                       // [1024] bucket start   (the list counts are not needed any more)
        uint32_t* s_cur = s_listcnt + 1024;                 // [1024] bucket cursor -> bucket end
        static_assert(kMaxScanGrid >= 2048 && kFinalThreads == 1024, "bucket order borrows s_listcnt as 2 x 1024 counters");
        uint32_t lo = 0xFFFFFFFFu, hi = 0u;
        for (uint32_t c = tid; c < nc; c += blockDim.x) { const uint32_t od = ent[c].od; lo = min(lo, od); hi = max(hi, od); }
        lo = __reduce_min_sync(0xFFFFFFFFu, lo);
        hi = __reduce_max_sync(0xFFFFFFFFu, hi);
        if (lane == 0) { atomicMin(&s_odlo, lo); atomicMax(&s_odhi, hi); }
        s_base[tid] = 0;
        __syncthreads();
        lo = s_odlo;
        const uint32_t range = s_odhi - lo;
        const uint32_t sh = range < 1024u ? 0u : 22u - (uint32_t)__clz(range);      // bucket = (od - lo) >> sh: monotone, at most 1023
        for (uint32_t c = tid; c < nc; c += blockDim.x) atomicAdd(&s_base[(ent[c].od - lo) >> sh], 1u);
        __syncthreads();
        {   // exclusive scan of the 1024 bucket sizes, one per thread
            const uint32_t v = s_base[tid];
            uint32_t incl = v;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, off);
                if ((int)lane >= off) incl += o;
            }
            if (lane == 31) s_warp[warp] = incl;
            __syncthreads();
            uint32_t before = 0;
            for (uint32_t w = 0; w < warp; ++w) before += s_warp[w];
            const uint32_t excl = before + incl - v;
            __syncthreads();
            s_base[tid] = excl;
            s_cur[tid] = excl;
        }
        __syncthreads();
        for (uint32_t c = tid; c < nc; c += blockDim.x) {
            const RerankEntry e = ent[c];
            ent2[atomicAdd(&s_cur[(e.od - lo) >> sh], 1u)] = e;
        }
        __syncthreads();
        for (uint32_t i = tid; i < nc; i += blockDim.x) {
            const RerankEntry me = ent2[i];
            const uint32_t b = (me.od - lo) >> sh;
            const uint32_t bs = s_base[b], be = s_cur[b];
            uint32_t pos = bs;
            for (uint32_t j = bs; j < be; ++j) pos += rerank_before(ent2[j], me) ? 1u : 0u;
            const float dist = dists[me.slot];
            const bool ok = (double)dist < p.max_dist;
            if (ok) local++;
            if (pos < p.k) {
                pbx_hit hh;
                if (ok) { hh.image_id = me.id; hh.dist = dist; hh.dot = dots[me.slot]; hh.norm2 = norms[me.slot]; hh.flags = 0; }
                else { hh.image_id = INT64_MAX; hh.dist = __int_as_float(0x7f800000); hh.dot = 0; hh.norm2 = 0; hh.flags = 0; }
                hits_g[pos] = hh;
            }
        }
    } else {
        block_sort_rerank(ent, n2);
        for (uint32_t c = tid; c < nc; c += blockDim.x) {
            const RerankEntry e = ent[c];
            const float dist = dists[e.slot];
            const bool ok = (double)dist < p.max_dist;
            if (ok) local++;
            if (c < p.k) {
                pbx_hit hh;
                if (ok) { hh.image_id = e.id; hh.dist = dist; hh.dot = dots[e.slot]; hh.norm2 = norms[e.slot]; hh.flags = 0; }
                else { hh.image_id = INT64_MAX; hh.dist = __int_as_float(0x7f800000); hh.dot = 0; hh.norm2 = 0; hh.flags = 0; }
                hits_g[c] = hh;
            }
        }
    }
    for (uint32_t c = nc + tid; c < p.k; c += blockDim.x) {
        pbx_hit hh; hh.image_id = INT64_MAX; hh.dist = __int_as_float(0x7f800000); hh.dot = 0; hh.norm2 = 0; hh.flags = 0;
        hits_g[c] = hh;
    }
    if (local) atomicAdd(&s_cnt, local);
    __syncthreads();
    if (s_excl) {
        // Paged search with candidates at or before the cursor: the certificate's kappa_k is that of the k-th best
        // SURVIVING candidate (by kappa).  buf is free again (ent is dead); the keys come back from the registers.
#pragma unroll
        for (uint32_t x = 0; x < kMaxKeep / kFinalThreads; ++x) {
            const uint32_t c = tid + x * kFinalThreads;
            if (c < nc && !((my_excl >> x) & 1u)) buf[atomicAdd(&s_scnt, 1u)] = my_key[x];
        }
        __syncthreads();
        const uint32_t ns = s_scnt;                            // nc - s_excl
        if (ns >= p.k) {
            if (ns > p.k) {
                TopBuf<u64> tk{buf, &s_scnt, &s_tau, p.cap, p.k};
                block_select_top(tk, &s_sel);
            }
            __shared__ u64 s_kmin;
            block_min_key(buf, p.k, &s_kmin, s_scratch64);
            if (tid == 0) s_kappa_k = key64_kappa(s_kmin);
        }
        __syncthreads();
    }

    PBX_FIN_STAMP(8);
    // ---- certificate (DESIGN.md section 5) ------------------------------------------------------------------
    if (tid == 0) {
        const uint32_t passing = s_cnt;
        *count_g = passing < p.k ? passing : p.k;
        SearchStatus st;
        st.n_candidates = nc;
        st.reserved = 0;
        st.need_exact = 0;
        st.theta = 0.0f;
        u64 searchable = p.n_allowed ? *p.n_allowed : (u64)p.n;
        // paged search: allowed rows at or below the cut (every row above it sorts before the cursor)
        if (cut_g) searchable -= min(searchable, (u64)*reinterpret_cast<const volatile uint32_t*>(&cut_g->above));
        if (searchable > nc) {                            // some (allowed, searchable) rows are not candidates
            const bool plateau_reachable = p.max_dist > (double)PBX_PLATEAU_DIST && s_nonplateau < p.k;
            const bool separated = (double)s_kappa_last < (double)s_kappa_k - (double)p.margin;
            const bool short_page = cut_g != nullptr && nc - s_excl < p.k;     // no k-th surviving candidate to bound with
            if (plateau_reachable || short_page) { st.need_exact = 1; st.theta = -__int_as_float(0x7f800000); }
            else if (!separated) { st.need_exact = 1; st.theta = (float)((double)s_kappa_k - (double)p.margin - 1e-7); }
        }
        if constexpr (BATCH) {
            if (p.boverflow[q]) { st.need_exact = 1; st.theta = -__int_as_float(0x7f800000); }   // candidates were dropped
        }
        *status_g = st;
        if constexpr (!BATCH) {
            p.tile_counter[0] = 0;                        // chunk scheduler
            p.tile_counter[32] = 0;                       // global bin threshold of the scan
            bool exact_follows = st.need_exact != 0;          // (without device-side launches the host has enqueued it already)
#ifdef PBX_USE_CDP
            if (st.need_exact) { __threadfence(); if (!launch_exact_tail(p.x)) { *count_g = PBX_COUNT_EXACT_LAUNCH_FAILED; exact_follows = false; } }
#endif
            if (p.done_flag && !exact_follows) {              // every hit was written before the barrier above
                __threadfence_system();
                *reinterpret_cast<volatile uint32_t*>(p.done_flag) = p.done_seq;
            }
        } else {
            // the last CTA to finish tail-launches the exact pass of every query that needs one, one after the
            // other (they share the scan scratch), from a single thread so that their order is well defined
            if (st.need_exact) atomicAdd(p.bticket + 1, 1u);      // bticket[1]: queries that need the exact pass (normally none)
            __threadfence();
            if (atomicAdd(p.bticket, 1u) == gridDim.x - 1) {
                *p.bticket = 0;
                __threadfence();
                const uint32_t n_need = *reinterpret_cast<volatile uint32_t*>(p.bticket + 1);
                p.bticket[1] = 0;
#ifdef PBX_USE_CDP
                for (uint32_t qq = 0; n_need && qq < p.nq; ++qq) {
                    if (*reinterpret_cast<volatile uint32_t*>(&p.status[qq].need_exact) == 0) continue;
                    ExactLaunch x = p.x;
                    x.scan.q16 += (size_t)qq * p.pitch;
                    x.scan.qbytes += (size_t)qq * p.pitch;
                    x.scan.qh += qq;
                    x.scan.status += qq;
                    if (x.scan.cut) x.scan.cut += qq;
                    x.fin.qbytes += (size_t)qq * p.pitch;
                    x.fin.hits += (size_t)qq * p.k;
                    x.fin.count += qq;
                    x.fin.status += qq;
                    if (!launch_exact_tail(x)) p.count[qq] = PBX_COUNT_EXACT_LAUNCH_FAILED;
                }
#endif
            }
        }
    }
}

}  // namespace pbx
