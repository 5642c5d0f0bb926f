// finalize.cuh -- everything around the scan: query preparation, the merge of the per-CTA
// candidate lists, kernel C (bit-exact f32 replay of the reference distance on the candidates,
// ordering by (dist, image_id), the `dist < max_dist` filter, LIMIT k) and the certificate that
// decides whether the exact pass must run.  Reference: src/engine.rs:375-383 (filter / order /
// limit), :572-588 (distance), :608-622 (f32 -> f64 widening before the comparison).
#pragma once
#include "scan.cuh"
#include "rerank.cuh"
#include "../../include/pixelbox_b200.h"

namespace pbx {

// ---- query preparation + seed of the scan's global threshold: one launch per query -----------------
// Every CTA centres the query into shared memory (c(q) = 2q - 255 as s16, zero in the row padding) and
// reduces sum c(q), sum c(q)^2; CTA 0 also writes them out for the scan / finalize kernels.
// Seed: a strided sample of the shard (gridDim.x * 256 rows: CTA b takes 256 consecutive rows starting at
// b * n / gridDim.x, one row per thread with 16 independent 16-byte loads in flight) is
// scored with the scan's integer arithmetic and counted in a private histogram; the last CTA to finish
// turns it into the bin b0 with at least `keep` sampled rows at or above it and stores it as the scan's
// starting global threshold.  b0 is a valid bound (sampled rows are real rows of the shard), so the scan's
// candidate buffers never see a flood of "everything passes" rows.  The private histogram is left zeroed.
struct PrepSeedParams {
    const uint8_t* query;       // raw [dim] bytes of this query
    uint32_t dim, pitch, pitch16;
    int16_t* q16;               // out [pitch]
    uint8_t* qbytes;            // out [pitch]
    QueryHeader* qh;            // out
    const uint4* rows;
    const float* inv_norm;
    uint32_t n;
    uint32_t keep;
    uint32_t do_seed;           // 0: gridDim.x == 1, the global threshold starts at 0
    uint32_t* seed_hist;        // [kHistBins], zero on entry and on exit
    uint32_t* ticket;           // zero on entry and on exit
    uint32_t* gbin;             // out: the scan's global bin threshold
    const uint32_t* allow;      // filtered search: only allowed sampled rows are counted (NULL = all).  With fewer than
                                // `keep` of them hist_threshold_warp gives 0: no starting threshold, which is valid
    const PageCut* cut;         // paged search: only sampled rows at or below the cut are counted (NULL = all)
};

__global__ void __launch_bounds__(kSeedThreads)
prep_seed_kernel(const PrepSeedParams p) {
    extern __shared__ __align__(16) unsigned char seed_smem[];
    int16_t* sq16 = reinterpret_cast<int16_t*>(seed_smem);           // [pitch] centred query
    __shared__ int ss[kSeedThreads / 32], sn[kSeedThreads / 32];
    __shared__ uint32_t s_last;
    __shared__ QueryHeader s_qh;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // No pdl_trigger() here on purpose: if the scan were launched early its CTAs would fill every SM while they
    // wait for this grid, and this grid waits for the previous query's finalize kernel *and its tail-launched
    // exact pass*, which needs those SMs: a deadlock.  The scan starts when this grid has completed.
    // Everything up to pdl_wait() reads only the caller's query and the immutable corpus, and writes only the
    // seed histogram / ticket (private to this kernel): it may overlap the previous query's finalize kernel.
    int s = 0, n2 = 0;
    for (uint32_t i = threadIdx.x; i < p.pitch; i += blockDim.x) {
        int c = 0;
        if (i < p.dim) c = centre(p.query[i]);
        sq16[i] = (int16_t)c;
        s += c;
        n2 += c * c;
    }
    for (int off = 16; off; off >>= 1) { s += __shfl_xor_sync(~0u, s, off); n2 += __shfl_xor_sync(~0u, n2, off); }
    if (lane == 0) { ss[warp] = s; sn[warp] = n2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int S = 0, N = 0;
        for (int w = 0; w < kSeedThreads / 32; ++w) { S += ss[w]; N += sn[w]; }
        QueryHeader h;
        h.sum_cq = S;
        h.norm2_q = N;
        h.inv_q = (float)(1.0 / sqrt((double)N));
        h.sa = 0.0f;
        s_qh = h;
    }
    __syncthreads();
    if (blockIdx.x == 0) {      // publish the query scratch only once the previous query's kernels are done with it
        pdl_wait();
        for (uint32_t i = threadIdx.x; i < p.pitch; i += blockDim.x) {
            p.q16[i] = sq16[i];
            p.qbytes[i] = i < p.dim ? p.query[i] : (uint8_t)0;
        }
        if (threadIdx.x == 0) {
            *p.qh = s_qh;
            if (!p.do_seed) *p.gbin = 0;
        }
    }
    if (!p.do_seed) return;

    const QueryHeader qh = s_qh;
    const uint32_t stride = p.n / gridDim.x;                        // >= 8 * 256 by the host's seeding condition
    {
        // one sampled row per thread, 16 independent 16-byte loads in flight (one DRAM round trip per 256 B of row)
        const uint32_t row = blockIdx.x * stride + threadIdx.x;
        const uint4* rp = p.rows + (size_t)row * p.pitch16;
        const int4* sq = reinterpret_cast<const int4*>(sq16);
        const uint4 zero = make_uint4(0, 0, 0, 0);
        int a = 0;
        for (uint32_t c0 = 0; c0 < p.pitch16; c0 += 16) {
            uint4 v[16];
#pragma unroll
            for (uint32_t i = 0; i < 16; ++i) v[i] = (c0 + i < p.pitch16) ? __ldg(rp + c0 + i) : zero;
#pragma unroll
            for (uint32_t i = 0; i < 16; ++i) {
                if (c0 + i < p.pitch16) {
                    const int4 x = sq[2 * (c0 + i)], y = sq[2 * (c0 + i) + 1];
                    const int qq[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
                    a = dot16(v[i], qq, a);
                }
            }
        }
        const int dot_i = 2 * a - 255 * qh.sum_cq;
        const float kappa = __fmul_rn(__fmul_rn((float)dot_i, __ldg(p.inv_norm + row)), qh.inv_q);
        if (row_allowed(p.allow, row) && kappa <= page_kappa_hi(p.cut)) atomicAdd(p.seed_hist + kappa_bin(kappa), 1u);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(p.ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x < 32) {
        const uint32_t b = hist_threshold_warp(p.seed_hist, p.keep, threadIdx.x);
        pdl_wait();             // the previous finalize kernel resets the global threshold: publish after it
        if (threadIdx.x == 0) { *p.gbin = b; *p.ticket = 0; }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < kHistBins; i += blockDim.x) p.seed_hist[i] = 0;
}

// ---- per-row metadata: inv_norm[r] = 1/sqrt(sum c(r_i)^2) and row_sum[r] = sum r_i, one warp per row ----------------------
// The one definition of both values: every path that writes a row (load, append, replace) computes them here.
__device__ __forceinline__ void row_meta_warp(const uint4* __restrict__ rows, uint32_t pitch16, uint32_t dim, uint64_t r, int lane,
                                              float* __restrict__ inv_norm, int* __restrict__ row_sum) {
    unsigned s1 = 0, s2 = 0;
    for (uint32_t c = lane; c < pitch16; c += 32) {
        uint4 v = __ldg(rows + r * pitch16 + c);
        s1 = dp4a_uu(v.x, 0x01010101u, s1); s1 = dp4a_uu(v.y, 0x01010101u, s1);
        s1 = dp4a_uu(v.z, 0x01010101u, s1); s1 = dp4a_uu(v.w, 0x01010101u, s1);
        s2 = dp4a_uu(v.x, v.x, s2); s2 = dp4a_uu(v.y, v.y, s2);
        s2 = dp4a_uu(v.z, v.z, s2); s2 = dp4a_uu(v.w, v.w, s2);
    }
    for (int off = 16; off; off >>= 1) { s1 += __shfl_xor_sync(~0u, s1, off); s2 += __shfl_xor_sync(~0u, s2, off); }
    if (lane == 0) {
        // sum (2v-255)^2 = 4 sum v^2 - 1020 sum v + 65025 d   (padding bytes are zero and excluded through d)
        long long n2 = 4ll * s2 - 1020ll * s1 + 65025ll * dim;
        inv_norm[r] = (float)(1.0 / sqrt((double)n2));
        row_sum[r] = (int)s1;                      // sum of the raw bytes: the batched (u8 x u8) path needs it per row
    }
}
__global__ void row_meta_kernel(const uint4* __restrict__ rows, uint32_t pitch16, uint32_t dim, uint64_t first, uint64_t n,
                                float* __restrict__ inv_norm, int* __restrict__ row_sum) {
    const uint64_t r = first + (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= first + n) return;
    row_meta_warp(rows, pitch16, dim, r, threadIdx.x & 31, inv_norm, row_sum);
}

// ---- synthetic corpus (bench/tests): same function as pixelbox_b200/synth.py ---------------------
__device__ __forceinline__ u64 splitmix64(u64 z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void synth_fill_kernel(uint8_t* __restrict__ rows, uint32_t pitch, uint32_t dim, uint64_t dst_row0, uint64_t n,
                                  u64 seed, u64 first_row, int64_t* __restrict__ ids) {
    const uint32_t chunks = pitch / 8;       // pitch is a multiple of 16
    const u64 total = n * chunks;
    for (u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (u64)gridDim.x * blockDim.x) {
        const u64 r = t / chunks;
        const uint32_t c = (uint32_t)(t % chunks);
        const u64 grow = first_row + r;
        const u64 rk = splitmix64(seed ^ (grow * 0xD1342543DE82EF95ull));
        u64 x = splitmix64(rk + c);
        const uint32_t b0 = c * 8;
        if (b0 >= dim) x = 0;
        else if (b0 + 8 > dim) x &= (~0ull) >> (8 * (b0 + 8 - dim));
        *reinterpret_cast<u64*>(rows + (dst_row0 + r) * pitch + b0) = x;
        if (c == 0) ids[dst_row0 + r] = (int64_t)(grow + 1);
    }
}

// ---- exact pass: merge of the per-CTA (dist, id) lists and output ----------------------------------
__global__ void __launch_bounds__(kFinalThreads, 1)
finalize_exact_kernel(const FinalizeExactParams p) {
    if (p.status->need_exact == 0) return;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    KeyX* buf = reinterpret_cast<KeyX*>(smem_raw);
    __shared__ uint32_t s_cnt, s_maxcnt;
    __shared__ KeyX s_tau;
    __shared__ uint32_t s_listcnt[kMaxScanGrid];
    if (threadIdx.x == 0) { s_cnt = 0; s_tau = KeyOps<KeyX>::lowest(); s_maxcnt = 0; }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < p.grid; b += blockDim.x) {
        uint32_t c = p.cand_cnt[b];
        s_listcnt[b] = c;
        atomicMax(&s_maxcnt, c);
    }
    __syncthreads();
    TopBuf<KeyX> tb{buf, &s_cnt, &s_tau, p.cap, p.k};
    const uint32_t total = s_maxcnt * p.grid;
    for (uint32_t base = 0; base < total; base += kMergeChunk) {
        if (s_cnt + kMergeChunk > p.cap) tb.compact();
        const KeyX tau = s_tau;
        __syncthreads();
#pragma unroll
        for (int x = 0; x < kMergeChunk / kFinalThreads; ++x) {
            const uint32_t e = base + x * kFinalThreads + threadIdx.x;
            bool pass = false;
            KeyX key = KeyOps<KeyX>::lowest();
            if (e < total) {
                const uint32_t rank = e / p.grid, b = e - rank * p.grid;
                if (rank < s_listcnt[b]) { key = p.cand[e]; pass = keyx_gt(key, tau); }
            }
            tb.push_warp(pass, key);
        }
        __syncthreads();
    }
    __syncthreads();
    tb.compact();
    const uint32_t nc = s_cnt < p.k ? s_cnt : p.k;
    for (uint32_t c = threadIdx.x; c < p.k; c += blockDim.x) {
        pbx_hit h;
        if (c < nc) {
            const KeyX key = buf[c];
            int idot = 0, inorm = 0;
            const uint8_t* row = p.rows + (size_t)key.row * p.pitch;
            for (uint32_t i = 0; i < p.dim; ++i) { int cr = centre(row[i]), cq = centre(p.qbytes[i]); idot += cq * cr; inorm += cr * cr; }
            h.image_id = keyx_id(key); h.dist = keyx_dist(key); h.dot = idot; h.norm2 = inorm; h.flags = 1;
        } else {
            h.image_id = INT64_MAX; h.dist = __int_as_float(0x7f800000); h.dot = 0; h.norm2 = 0; h.flags = 0;
        }
        p.hits[c] = h;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        *p.count = nc;
        *p.tile_counter = 0;
        atomicAdd(p.exact_passes, 1ull);
        if (p.done_flag) {
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t*>(p.done_flag) = p.done_seq;
        }
    }
}

// ---- merge after the all-gather (SURVEY.md 8e), device side ----------------------------------------
// gathered: [n_shards][nq][k] hits, counts: [n_shards][nq]; every shard list is ordered by
// (dist, image_id).  One thread per gathered element computes its global rank as the number of
// elements of all lists that precede it under (dist, image_id, shard) -- a binary search per list --
// and writes itself to out[rank] if rank < k.  n_shards * k is at most a few thousand.
__device__ __forceinline__ bool hit_before(const pbx_hit& a, uint32_t sa, const pbx_hit& b, uint32_t sb) {
    if (a.dist != b.dist) return a.dist < b.dist;
    if (a.image_id != b.image_id) return a.image_id < b.image_id;
    return sa < sb;
}
// L2-coherent read of a record: used for mailboxes that peer GPUs write over NVLink (L1 is not coherent with them)
__device__ __forceinline__ pbx_hit ld_hit_cg(const pbx_hit* p) {
    const unsigned long long* w = reinterpret_cast<const unsigned long long*>(p);
    const unsigned long long a = __ldcg(w), b = __ldcg(w + 1), c = __ldcg(w + 2);
    pbx_hit h;
    h.image_id = (int64_t)a;
    h.dist = __uint_as_float((uint32_t)(b & 0xFFFFFFFFull));
    h.dot = (int32_t)(b >> 32);
    h.norm2 = (int32_t)(c & 0xFFFFFFFFull);
    h.flags = (uint32_t)(c >> 32);
    return h;
}

// One CTA merges the n_shards lists of query q (gathered is [n_shards][nq][k]); counts may be NULL.
// The order keys (dist, image_id) of all lists are staged in shared memory first when they fit (kMergeSmemKeys),
// so that the n_shards * log2(k) probes per record are shared-memory reads and not dependent L2 round trips
// (at 8 shards x 100 records the L2 version spent ~50 us in ~220 serial probes per thread).
constexpr uint32_t kMergeThreads = 512;
constexpr uint32_t kMergeSmemKeys = 8192;                       // 12 B per key -> 96 KB of dynamic shared memory
__host__ __device__ inline uint32_t merge_smem_bytes(uint32_t n_shards, uint32_t k) {
    const uint64_t keys = (uint64_t)n_shards * k;
    return keys <= kMergeSmemKeys ? (uint32_t)(keys * 12u) : 0u;
}
__device__ __forceinline__ bool key_before(uint32_t da, long long ia, uint32_t sa, uint32_t db, long long ib, uint32_t sb) {
    if (da != db) return da < db;
    if (ia != ib) return ia < ib;
    return sa < sb;
}

__device__ inline void merge_hits_block(const pbx_hit* gathered, const uint32_t* counts, uint32_t n_shards, uint32_t nq, uint32_t k,
                                        uint32_t q, pbx_hit* out, uint32_t* out_count, unsigned char* stage) {
    __shared__ uint32_t s_cnt[PBX_MAX_SHARDS];
    __shared__ uint32_t s_total;
    const uint32_t total = n_shards * k;
    long long* s_id = reinterpret_cast<long long*>(stage);
    uint32_t* s_dist = reinterpret_cast<uint32_t*>(stage + (size_t)total * 8u);
    if (threadIdx.x == 0) s_total = 0;
    if (stage) {
        for (uint32_t e = threadIdx.x; e < total; e += blockDim.x) {
            const uint32_t s = e / k, i = e - s * k;
            const pbx_hit h = ld_hit_cg(gathered + ((size_t)s * nq + q) * k + i);
            s_id[e] = h.image_id;
            s_dist[e] = ord_f32(h.dist);
        }
    }
    __syncthreads();
    const uint32_t ord_inf = ord_f32(__int_as_float(0x7f800000));
    for (uint32_t s = threadIdx.x; s < n_shards; s += blockDim.x) {
        uint32_t c;
        if (counts) {
            c = min(counts[s * nq + q], k);
        } else {                                    // unused tail slots carry dist = +inf: count the finite prefix
            const pbx_hit* list = gathered + ((size_t)s * nq + q) * k;
            uint32_t lo = 0, hi = k;
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                const bool finite = stage ? (s_dist[s * k + mid] < ord_inf) : (ld_hit_cg(list + mid).dist < __int_as_float(0x7f800000));
                if (finite) lo = mid + 1; else hi = mid;
            }
            c = lo;
        }
        s_cnt[s] = c;
        atomicAdd(&s_total, c);
    }
    __syncthreads();
    const uint32_t n_out = min(s_total, k);
    for (uint32_t e = threadIdx.x; e < total; e += blockDim.x) {
        const uint32_t s = e / k, i = e - s * k;
        if (i >= s_cnt[s]) continue;
        uint32_t rank = 0;
        if (stage) {
            const uint32_t md = s_dist[e];
            const long long mi = s_id[e];
            for (uint32_t t = 0; t < n_shards && rank < k; ++t) {
                if (t == s) { rank += i; continue; }         // its own list is already ordered
                uint32_t lo = 0, hi = s_cnt[t];
                while (lo < hi) {                   // first element of list t that does not precede this record
                    const uint32_t mid = (lo + hi) >> 1;
                    if (key_before(s_dist[t * k + mid], s_id[t * k + mid], t, md, mi, s)) lo = mid + 1; else hi = mid;
                }
                rank += lo;
            }
            if (rank < k) out[(size_t)q * k + rank] = ld_hit_cg(gathered + ((size_t)s * nq + q) * k + i);
        } else {
            const pbx_hit me = ld_hit_cg(gathered + ((size_t)s * nq + q) * k + i);
            for (uint32_t t = 0; t < n_shards; ++t) {
                if (t == s) { rank += i; continue; }
                const pbx_hit* list = gathered + ((size_t)t * nq + q) * k;
                uint32_t lo = 0, hi = s_cnt[t];
                while (lo < hi) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (hit_before(ld_hit_cg(list + mid), t, me, s)) lo = mid + 1; else hi = mid;
                }
                rank += lo;
            }
            if (rank < k) out[(size_t)q * k + rank] = me;
        }
    }
    for (uint32_t i = n_out + threadIdx.x; i < k; i += blockDim.x) {
        pbx_hit h; h.image_id = INT64_MAX; h.dist = __int_as_float(0x7f800000); h.dot = 0; h.norm2 = 0; h.flags = 0;
        out[(size_t)q * k + i] = h;
    }
    if (threadIdx.x == 0) out_count[q] = n_out;
}

__global__ void __launch_bounds__(kMergeThreads)
merge_hits_kernel(const pbx_hit* __restrict__ gathered, const uint32_t* __restrict__ counts, uint32_t n_shards,
                  uint32_t nq, uint32_t k, pbx_hit* __restrict__ out, uint32_t* __restrict__ out_count, uint32_t stage_bytes) {
    extern __shared__ __align__(16) unsigned char merge_stage[];
    merge_hits_block(gathered, counts, n_shards, nq, k, blockIdx.x, out, out_count, stage_bytes ? merge_stage : nullptr);
}

// ---- the exchange step fused with the merge, over NVLink peer memory (SURVEY.md 8e) -----------------------
// Every rank owns a mailbox (two slots of [world][nq][k] records) and a flag array, both mapped into its peers'
// address spaces (CUDA IPC).  One CTA per query: it posts this rank's k records straight into the mailbox of every
// peer (plain stores to peer addresses), publishes them with a system-scope release of a per-(query, source)
// sequence flag, spins with acquire loads until all `world` flags of its own mailbox carry this call's sequence
// number, and merges the lists under (dist, image_id).  No NCCL call, no host step: post, signal, wait and merge
// are one kernel on the search stream.  Slots alternate per call: a rank can be at most one call ahead of its
// slowest peer (it cannot finish call i+1 before that peer has posted i+1, i.e. finished reading call i).
struct ExchangeParams {
    pbx_hit* peer_mail[PBX_MAX_SHARDS];   // mailbox base of every rank (slot 0), as mapped in this process
    uint32_t* peer_flag[PBX_MAX_SHARDS];  // flag base of every rank
    const pbx_hit* local;                 // [nq][k] this rank's hits
    pbx_hit* out;                         // [nq][k]
    uint32_t* out_count;                  // [nq]
    uint32_t rank, world, nq, k;
    uint32_t slot, seq;
    uint32_t slot_records;                // records per mailbox slot
    uint32_t slot_flags;                  // flags per slot (max_queries * world)
    uint32_t stage_bytes;                 // dynamic shared memory for the merge keys (0: probe through L2)
    // zero-copy completion of a one-query host call (NULL otherwise): out / out_count are host-mapped, the shard's own
    // count (which may carry an error marker) is copied next to them, and done_seq is published last
    const uint32_t* local_count;
    uint32_t* local_count_out;
    uint32_t* done_flag;
    uint32_t done_seq;
};

__global__ void __launch_bounds__(kMergeThreads)
exchange_merge_kernel(const __grid_constant__ ExchangeParams p) {
    extern __shared__ __align__(16) unsigned char merge_stage[];
    const uint32_t q = blockIdx.x;
    __shared__ uint32_t s_timeout;
    if (threadIdx.x == 0) s_timeout = 0;
    __syncthreads();
    // 1. post
    const unsigned long long* src = reinterpret_cast<const unsigned long long*>(p.local + (size_t)q * p.k);
    const uint32_t words = p.k * 3u;                                            // 24-byte records as 8-byte words
    for (uint32_t peer = 0; peer < p.world; ++peer) {
        unsigned long long* dst = reinterpret_cast<unsigned long long*>(
            p.peer_mail[peer] + (size_t)p.slot * p.slot_records + ((size_t)p.rank * p.nq + q) * p.k);
        for (uint32_t i = threadIdx.x; i < words; i += blockDim.x) dst[i] = src[i];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < p.world) {
        uint32_t* f = p.peer_flag[threadIdx.x] + (size_t)p.slot * p.slot_flags + (size_t)q * p.world + p.rank;
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(f), "r"(p.seq) : "memory");
    }
    // 2. wait for the records of all ranks for this query
    if (threadIdx.x < p.world) {
        const uint32_t* f = p.peer_flag[p.rank] + (size_t)p.slot * p.slot_flags + (size_t)q * p.world + threadIdx.x;
        uint32_t v;
        const long long t0 = clock64();
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            // a peer that died must not hang this GPU for ever: give up after ~10 s and flag the result
            if (v != p.seq && clock64() - t0 > (20ll << 30)) { atomicOr(&s_timeout, 1u); break; }
        } while (v != p.seq);
    }
    __syncthreads();
    // 3. merge from this rank's own mailbox (records were written by peers: read through L2)
    merge_hits_block(p.peer_mail[p.rank] + (size_t)p.slot * p.slot_records, nullptr, p.world, p.nq, p.k, q, p.out, p.out_count,
                     p.stage_bytes ? merge_stage : nullptr);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_timeout) p.out_count[q] = 0xFFFFFFFFu;                          // "exchange timed out" marker for the host
        if (p.done_flag) {                                                    // (one query = one CTA: no counting needed)
            p.local_count_out[q] = p.local_count[q];
            __threadfence_system();
            *reinterpret_cast<volatile uint32_t*>(p.done_flag) = p.done_seq;
        }
    }
}

// ---- the ingest quantizer (src/image_hashes/efficientnet.rs:39), SURVEY.md 8f N3 --------------------------
//   128u8.saturating_add_signed((f * 128.0f32).max(-128.0f32).min(128.0f32) as i8)
// `as i8` truncates toward zero and saturates (so +128.0 -> 127); f32::max returns the other operand for a NaN,
// so NaN -> -128 -> byte 0.  Note the asymmetry the reference lives with: this encoder is centred on 128, the
// decoder of cosine_distance on 127.5 (src/engine.rs:576); both are kept bit-compatible, not "fixed".
__global__ void quantize_kernel(const float* __restrict__ in, uint64_t n, uint8_t* __restrict__ out) {
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        float x = __fmul_rn(in[i], 128.0f);
        x = fmaxf(x, -128.0f);              // fmaxf(NaN, a) == a, like f32::max
        x = fminf(x, 128.0f);
        const int v = x >= 127.0f ? 127 : (x <= -128.0f ? -128 : (int)x);      // (int) truncates toward zero
        out[i] = (uint8_t)(128 + v);
    }
}

// ---- cosine_distance for explicit pairs (src/engine.rs:572-588 as a batch) -------------------------
__global__ void pair_distance_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint64_t n, uint32_t dim,
                                     float* __restrict__ out_dist, int* __restrict__ out_dot, int* __restrict__ out_na,
                                     int* __restrict__ out_nb) {
    __shared__ float lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = ref_decode(i);
    __syncthreads();
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint8_t* pa = a + t * dim;
    const uint8_t* pb = b + t * dim;
    float sa = 0.0f, sb = 0.0f, dot = 0.0f;
    int idot = 0, ina = 0, inb = 0;
    for (uint32_t i = 0; i < dim; ++i) { float x = lut[pa[i]]; sa = ref_fold(sa, x, x); int c = centre(pa[i]); ina += c * c; }
    for (uint32_t i = 0; i < dim; ++i) { float y = lut[pb[i]]; sb = ref_fold(sb, y, y); int c = centre(pb[i]); inb += c * c; }
    for (uint32_t i = 0; i < dim; ++i) { dot = ref_fold(dot, lut[pa[i]], lut[pb[i]]); idot += centre(pa[i]) * centre(pb[i]); }
    out_dist[t] = ref_distance(sa, sb, dot);
    if (out_dot) out_dot[t] = idot;
    if (out_na) out_na[t] = ina;
    if (out_nb) out_nb[t] = inb;
}

// ---- byte_distance (src/engine.rs:590-592) and hamming_distance (:594-604) for explicit pairs, SURVEY.md 8f N4 ------
// One warp per pair; 4 bytes per lane and step (__vsadu4 = sum of absolute byte differences, __popc of the xor) when
// dim is a multiple of 4, bytes otherwise.  Both sums are exact integers; the reference's f32 fold of |a - b| is exact
// too (every partial sum is an integer below 2^24), so one correctly rounded division reproduces it bit for bit.
// hamming_distance sums per-byte bit counts in a u8 upstream: the sum wraps modulo 256 in a release build, which is
// what `out_ham` reproduces; `out_bits` is the true count.
__global__ void __launch_bounds__(256)
pair_byte_hamming_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint64_t n, uint32_t dim,
                         float* __restrict__ out_byte, uint32_t* __restrict__ out_l1, float* __restrict__ out_ham,
                         uint32_t* __restrict__ out_bits) {
    const uint64_t pair = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (pair >= n) return;
    const uint8_t* pa = a + pair * dim;
    const uint8_t* pb = b + pair * dim;
    uint32_t l1 = 0, bits = 0;
    if ((dim & 3u) == 0 && (((uintptr_t)a | (uintptr_t)b) & 3u) == 0) {
        const uint32_t* wa = reinterpret_cast<const uint32_t*>(pa);
        const uint32_t* wb = reinterpret_cast<const uint32_t*>(pb);
        for (uint32_t i = lane; i < dim / 4; i += 32) {
            const uint32_t x = wa[i], y = wb[i];
            l1 += __vsadu4(x, y);
            bits += (uint32_t)__popc(x ^ y);
        }
    } else {
        for (uint32_t i = lane; i < dim; i += 32) {
            const int x = pa[i], y = pb[i];
            l1 += (uint32_t)abs(x - y);
            bits += (uint32_t)__popc((uint32_t)(x ^ y));
        }
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        l1 += __shfl_xor_sync(0xFFFFFFFFu, l1, off);
        bits += __shfl_xor_sync(0xFFFFFFFFu, bits, off);
    }
    if (lane == 0) {
        if (out_byte) out_byte[pair] = __fdiv_rn((float)l1, __fmul_rn(255.0f, (float)dim));
        if (out_l1) out_l1[pair] = l1;
        if (out_ham) out_ham[pair] = __fdiv_rn((float)(bits & 0xFFu), __fmul_rn(8.0f, (float)dim));
        if (out_bits) out_bits[pair] = bits;
    }
}

}  // namespace pbx
