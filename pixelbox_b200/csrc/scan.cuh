// scan.cuh -- kernel A: the HBM-bound single-query scan (replaces the per-row SQLite -> UDF ->
// cosine_distance loop of src/engine.rs:375-383 / :608-622 / :572-588 in the reference).
//
// One persistent CTA grid streams the row-major u8 corpus once.  L lanes share a row (16-byte
// coalesced ld.global.nc per lane), the query lives in registers as centred 16-bit values
// c(q) = 2q - 255, and IDP.2A (dp2a) accumulates  acc = sum c(q_i) * r_i  exactly in int32, so
//     dot_i = sum c(q_i) c(r_i) = 2 * acc - 255 * sum c(q_i)
// needs no per-row sum.  A transposing butterfly (L-1 shuffles per L rows) leaves one finished
// row per lane; the ranking key is kappa = dot_i / sqrt(norm2_q * norm2_r) in f32 using the
// per-row 1/sqrt(norm2_r) precomputed at load time (4 bytes per row, the only metadata read).
// Rows that beat the CTA's running threshold are pushed into a shared-memory buffer; the buffer
// is sorted and cut back to `keep` entries when it runs out of headroom (rare after warm-up).
//
// EXACT = false: fast pass, key = (kappa, row), keep = k + slack candidates per CTA.
// EXACT = true : tie-resolving pass.  Rows with kappa >= theta are replayed with the
//                reference's f32 arithmetic in-kernel and ranked by the exact (dist, image_id);
//                launched after every fast pass and exits at once unless the fast pass could
//                not certify its answer (status->need_exact).
#pragma once
#include "common.cuh"

namespace pbx {

struct QueryHeader {            // written by prep_query_kernel (+ sa by the finalize kernel)
    int sum_cq;                 // sum c(q_i), i < dim
    int norm2_q;                // sum c(q_i)^2
    float inv_q;                // 1/sqrt(norm2_q), f32-rounded from f64
    float sa;                   // reference's sequential f32 fold of the decoded query (engine.rs:580)
};

struct SearchStatus {           // one per query, written by the finalize kernel
    uint32_t need_exact;        // 1: the certificate failed, the exact pass must run
    float theta;                // exact pass replays rows with kappa >= theta
    uint32_t n_candidates;
    uint32_t reserved;
};

struct ScanParams {
    const uint4* rows;          // [capacity][pitch16] u8 rows, zero padded to a multiple of 16 bytes
    const float* inv_norm;      // [capacity] 1/sqrt(norm2_r)
    const int64_t* ids;         // [capacity]
    uint32_t n;                 // committed rows visible to this search
    uint32_t pitch16;           // row pitch in 16-byte chunks
    uint32_t dim;
    float max_dist;             // EXACT only: the smallest f32 >= the caller's f64 max_dist (dist < it <=> dist < max_dist)
    const int16_t* q16;         // [pitch] centred query, zero in the padding
    const uint8_t* qbytes;      // [pitch] raw query bytes
    const QueryHeader* qh;
    uint32_t keep;              // entries kept per CTA (k + slack, or k for EXACT)
    uint32_t cap;               // shared buffer capacity, power of two >= keep + kTileRows
    void* cand;                 // [keep][grid] keys, rank-major (u64 or KeyX)
    uint32_t* cand_cnt;         // [grid]
    uint32_t* tile_counter;     // dynamic tile scheduler (reset by the finalize kernel)
    uint32_t* hist;             // [kHistBins] fast pass: kappa histogram of every pushed key (global + merge threshold)
    const SearchStatus* status; // EXACT only
    PageCut* cut;               // paged search: this query's cut and cursor (page.cuh), NULL = first page; the fast pass
                                // reads it only in its RESTRICT instantiations and adds the rows above the cut to cut->above
    const uint32_t* allow;      // filtered search: bit per row (row_allowed), NULL = every row; the fast pass reads it
                                // only in its RESTRICT instantiations
};
// 128 bytes, and every field the unrestricted fast pass reads at the offset it had before paged searches: a larger
// parameter block changes how the compiler reads it (and the fast pass's code)
static_assert(sizeof(ScanParams) == 128, "ScanParams layout");

// 16 corpus bytes against 16 centred query values: 8 x IDP.2A
__device__ __forceinline__ int dot16(const uint4& v, const int* q, int acc) {
    acc = dp2a_lo(q[0], v.x, acc); acc = dp2a_hi(q[1], v.x, acc);
    acc = dp2a_lo(q[2], v.y, acc); acc = dp2a_hi(q[3], v.y, acc);
    acc = dp2a_lo(q[4], v.z, acc); acc = dp2a_hi(q[5], v.z, acc);
    acc = dp2a_lo(q[6], v.w, acc); acc = dp2a_hi(q[7], v.w, acc);
    return acc;
}

// L lanes each hold L partial sums (one per row); afterwards lane j holds the full sum of row j.
template <int L>
__device__ __forceinline__ int transpose_reduce(int (&acc)[L], int j) {
#pragma unroll
    for (int off = L / 2; off >= 1; off >>= 1) {
        const bool up = (j & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            int send = up ? acc[i] : acc[i + off];
            int keep = up ? acc[i + off] : acc[i];
            acc[i] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, off);
        }
    }
    return acc[0];
}

// Bit-exact replay of the reference's row norm and dot folds for one row (src/engine.rs:580, :585),
// strictly in element order.  The row is read with 16-byte loads, one batch of four prefetched ahead
// of the arithmetic; q (raw bytes) and q16 (centred s16) may live in shared or global memory.
// The exact integers come from the same bytes: dot_i = 2 * sum c(q) r - 255 * sum c(q),
// norm2 = 4 sum r^2 - 1020 sum r + 65025 d (row padding is zero, q16 padding is zero).
struct ReplayOut {
    float sb, dot;
    int idot, inorm;
};

__device__ __forceinline__ void replay_bytes(uint32_t rv, uint32_t qv, int nbytes, const float* lut, float& s, float& d) {
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        if (b < nbytes) {
            const float fb = lut[(rv >> (8 * b)) & 255u], fa = lut[(qv >> (8 * b)) & 255u];
            s = ref_fold(s, fb, fb);
            d = ref_fold(d, fa, fb);
        }
    }
}

template <bool WITH_INTS>
__device__ __forceinline__ ReplayOut replay_row(const uint8_t* __restrict__ row, const uint8_t* q, const int16_t* q16, uint32_t dim,
                                                int sum_cq, const float* lut) {
    const uint4* r4 = reinterpret_cast<const uint4*>(row);
    const uint32_t* q32 = reinterpret_cast<const uint32_t*>(q);
    const int4* q16v = reinterpret_cast<const int4*>(q16);
    const uint32_t full = dim >> 4, chunks = (dim + 15) >> 4;
    float s = 0.0f, d = 0.0f;
    int acc = 0;
    unsigned s1 = 0, s2 = 0;
    const uint4 zero = make_uint4(0, 0, 0, 0);
    uint4 cur[4], nxt[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) cur[i] = ((uint32_t)i < chunks) ? __ldg(r4 + i) : zero;
    for (uint32_t c = 0; c < chunks; c += 4) {
#pragma unroll
        for (int i = 0; i < 4; ++i) nxt[i] = (c + 4 + i < chunks) ? __ldg(r4 + c + 4 + i) : zero;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t ci = c + i;
            if (ci < chunks) {
                const uint4 v = cur[i];
                if (ci < full) {
                    replay_bytes(v.x, q32[4 * ci + 0], 4, lut, s, d);
                    replay_bytes(v.y, q32[4 * ci + 1], 4, lut, s, d);
                    replay_bytes(v.z, q32[4 * ci + 2], 4, lut, s, d);
                    replay_bytes(v.w, q32[4 * ci + 3], 4, lut, s, d);
                } else {                            // ragged tail: dim is not a multiple of 16
                    const int rem = (int)(dim - (ci << 4));
                    replay_bytes(v.x, q32[4 * ci + 0], rem, lut, s, d);
                    replay_bytes(v.y, q32[4 * ci + 1], rem - 4, lut, s, d);
                    replay_bytes(v.z, q32[4 * ci + 2], rem - 8, lut, s, d);
                    replay_bytes(v.w, q32[4 * ci + 3], rem - 12, lut, s, d);
                }
                if constexpr (WITH_INTS) {
                    const int4 a = q16v[2 * ci], b = q16v[2 * ci + 1];
                    const int qq[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                    acc = dot16(v, qq, acc);
                    s1 = dp4a_uu(v.x, 0x01010101u, s1); s1 = dp4a_uu(v.y, 0x01010101u, s1);
                    s1 = dp4a_uu(v.z, 0x01010101u, s1); s1 = dp4a_uu(v.w, 0x01010101u, s1);
                    s2 = dp4a_uu(v.x, v.x, s2); s2 = dp4a_uu(v.y, v.y, s2);
                    s2 = dp4a_uu(v.z, v.z, s2); s2 = dp4a_uu(v.w, v.w, s2);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) cur[i] = nxt[i];
    }
    ReplayOut o;
    o.sb = s;
    o.dot = d;
    o.idot = 2 * acc - 255 * sum_cq;
    o.inorm = (int)(4u * s2 - 1020u * s1 + 65025u * dim);
    return o;
}

#ifdef PBX_EXP_PROFILE
// experiment builds only: per-CTA counters of the fast pass
// [0] pushes  [1] compactions  [2] cycles waiting at rendezvous  [3] cycles in compaction  [4] total cycles
// [5] entries before the final filter  [6] entries after it  [7] chunks processed
__device__ unsigned long long g_scan_prof[kMaxScanGrid][8];
#define PBX_PROF_ADD(i, v) do { if (threadIdx.x == 0) g_scan_prof[blockIdx.x][i] += (unsigned long long)(v); } while (0)
#else
#define PBX_PROF_ADD(i, v) do { } while (0)
#endif

template <typename K, bool EXACT>
struct ScanShared {
    uint32_t cnt;
    uint32_t done;              // warps that have run out of work
    uint32_t gb;                // CTA copy of the global bin threshold (polled by warp 0 only: one hot line, few readers)
    uint32_t tile[2];           // generic kernel: tile index broadcast
    K tau;
    float lut[EXACT ? 256 : 1];
    SelectScratch sel;
};

constexpr int scan_minb(int pitch16) { return pitch16 >= 16 ? 2 : 4; }

// Fast shapes: pitch16 == L * C, L lanes per row, C chunks per lane.  RAGGED: the same lane layout for any
// pitch16 <= L * C (row stride taken from the parameters, lane slots beyond the row neither load nor count), so
// that every row length streams with coalesced 16-byte loads; only the idle slots are lost.
// RESTRICT (fast pass only): a filtered and/or paged search.  A row is pushed -- and so counted in the histograms every
// threshold comes from -- only if its bit in p.allow is set (when there is a filter) and its kappa is at most the cut
// (when there is a cursor).  The 32 rows of a warp iteration are consecutive: one broadcast bitmap word per iteration.
// Allowed rows above the cut are counted (one ballot per warp iteration, one atomic per chunk) for the certificate's
// trivially-exact case.  A template flag, so that the unrestricted instantiations are the same code as before.  The
// exact pass tests p.allow and the cut at run time, before the replay of a row, and drops the rows at or before the
// cursor after it.
template <int L, int C, bool EXACT, int MINB = scan_minb(L * C), bool RAGGED = false, bool RESTRICT = false>
__global__ void __launch_bounds__(kScanThreads, MINB)
scan_kernel(const ScanParams p) {
    static_assert(!(RESTRICT && EXACT), "the exact pass tests the filter and the cut at run time");
    using K = typename std::conditional<EXACT, KeyX, u64>::type;
    constexpr int G = 32 / L;                 // rows handled by one warp-wide load
    constexpr int P16 = L * C;                // row pitch in chunks (compile time for fast shapes)
    const uint32_t PR = RAGGED ? p.pitch16 : (uint32_t)P16;       // actual row stride in chunks
    extern __shared__ __align__(16) unsigned char smem_raw[];
    K* buf = reinterpret_cast<K*>(smem_raw);
    __shared__ ScanShared<K, EXACT> sh;

    pdl_wait();                 // the query preparation / threshold seed (and everything before it) is complete
    pdl_trigger();              // the finalize kernel may be scheduled as soon as an SM has room for it
    if constexpr (EXACT) {
        if (p.status->need_exact == 0) return;
        sh.lut[threadIdx.x & 255] = ref_decode(threadIdx.x & 255);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane / L, j = lane % L;
#ifdef PBX_EXP_PROFILE
    const long long t_kernel0 = clock64();
#endif

    // centred query chunks of this lane: chunk index j + c*L, 16 values = 8 packed registers each
    int q[C][8];
    bool has_chunk[C];
    uint32_t coff[C];                           // RAGGED: chunk offset of slot c within the row
#pragma unroll
    for (int c = 0; c < C; ++c) {
        has_chunk[c] = !RAGGED || (uint32_t)(j + c * L) < PR;
        coff[c] = has_chunk[c] ? (uint32_t)(j + c * L) : PR - 1u;
        const int4* src = reinterpret_cast<const int4*>(p.q16 + (size_t)(has_chunk[c] ? (j + c * L) : 0) * 16);
        int4 a = __ldg(src), b = __ldg(src + 1);
        if (!has_chunk[c]) { a = make_int4(0, 0, 0, 0); b = a; }
        q[c][0] = a.x; q[c][1] = a.y; q[c][2] = a.z; q[c][3] = a.w;
        q[c][4] = b.x; q[c][5] = b.y; q[c][6] = b.z; q[c][7] = b.w;
    }
    const QueryHeader qh = *p.qh;
    const int bias = -255 * qh.sum_cq;
    float theta = 0.0f;
    if constexpr (EXACT) theta = p.status->theta;
    float cut = __int_as_float(0x7f800000);
    if constexpr (EXACT || RESTRICT) cut = page_kappa_hi(p.cut);

    uint32_t* const gbin = p.tile_counter + 32;        // its own 128-byte line, away from the chunk counter
    // sh.gb starts at the global bin threshold seeded by prep_seed_kernel from a strided sample of the shard (fast pass)
    if (threadIdx.x == 0) { sh.cnt = 0; sh.done = 0; sh.gb = EXACT ? 0u : *reinterpret_cast<volatile uint32_t*>(gbin); sh.tau = KeyOps<K>::lowest(); }
    TopBuf<K> tb{buf, &sh.cnt, &sh.tau, p.cap, p.keep};
    __syncthreads();

    // Global threshold (fast pass): every pushed key is also counted in a global histogram over kappa.
    // At geometrically spaced claim numbers the claiming warp scans the histogram for the highest bin b*
    // with at least `keep` entries at or above it and publishes it (atomicMax): rows below b* cannot be
    // among the best `keep` of the whole shard, whichever CTA sees them.  After the first few chunks the
    // push rate is ~keep / rows-seen-by-all-CTAs, so buffers almost never need cutting back mid-scan.
    uint32_t gb = sh.gb;                               // (published before the barrier above)
    const uint32_t total_warps = gridDim.x * kScanWarps;

    // Warp-autonomous scheduling: every warp claims chunks of kChunkRows rows from a global counter
    // (GRAB chunks per atomic, the next claim is in flight while the current one is processed) and never
    // waits for its siblings in the steady state.  The CTA only meets at a barrier when the candidate
    // buffer is within one round of pushes of its capacity (cut back to `keep`) or when every warp has
    // run out of work.  A warp that starts a chunk has seen cnt <= threshold, so at most
    // kScanWarps * kChunkRows = kTileRows pushes can follow: cap >= threshold + kTileRows.
    constexpr uint32_t GRAB = (P16 >= 16) ? 1u : 16u / P16;
    const uint32_t n_chunks = (p.n + kChunkRows - 1) / kChunkRows;
    const uint32_t threshold = p.cap - kTileRows;
    uint32_t cur = 0, end = 0, nxt = 0;
    if (lane == 0) nxt = atomicAdd(p.tile_counter, GRAB);
    bool counted = false;
    for (;;) {
        if (cur == end && !counted) {
            cur = __shfl_sync(0xFFFFFFFFu, nxt, 0);
            end = cur + GRAB;
            if (lane == 0 && cur < n_chunks) nxt = atomicAdd(p.tile_counter, GRAB);
            if constexpr (!EXACT) {
                const uint32_t claim = cur / GRAB;
                if (cur < n_chunks && claim >= total_warps && claim % total_warps == 0 &&
                    ((claim / total_warps) & (claim / total_warps - 1)) == 0) {
                    const uint32_t b = hist_threshold_warp(p.hist, p.keep, lane);
                    if (lane == 0 && b) { atomicMax(gbin, b); atomicMax(&sh.gb, b); }
                }
            }
        }
        const bool have = cur < n_chunks;
        if (have && *reinterpret_cast<volatile uint32_t*>(&sh.cnt) <= threshold) {
            const K tau = sh.tau;
            const uint32_t chunk_row0 = cur * kChunkRows;
            ++cur;
            uint32_t gpoll = 0;
            uint32_t n_above = 0;                       // RESTRICT: allowed rows of this chunk above the cut
            if constexpr (!EXACT) {
                // warp 0 polls the global word once per chunk (consumed at the end of the chunk, so the L2 round
                // trip is hidden) and republishes it in shared memory for its siblings
                if (warp == 0 && lane == 0) gpoll = *reinterpret_cast<volatile uint32_t*>(gbin);
            }
            constexpr int UNR = (L * C >= 16) ? 1 : kItersPerChunk;
#pragma unroll UNR
            for (int it = 0; it < kItersPerChunk; ++it) {
                const uint32_t row0 = chunk_row0 + (uint32_t)it * kRowsPerWarpIter;
                const uint32_t my_row = row0 + (uint32_t)(j * G + g);
                uint32_t allow_word = ~0u;
                if constexpr (RESTRICT) {
                    if (p.allow) allow_word = __ldg(p.allow + (row0 >> 5));   // rows [row0, row0 + 32), row0 % 32 == 0
                }
                float gthr = -__int_as_float(0x7f800000);
                uint32_t gb_new = 0;
                if constexpr (!EXACT) {
                    gthr = bin_threshold(gb);
                    gb_new = *reinterpret_cast<volatile uint32_t*>(&sh.gb);  // refreshed every 32 rows; used by the next iteration
                }
#ifdef PBX_EXP_NOMETA
                const float inv_r = 1.0e-4f;
#else
                const float inv_r = __ldg(p.inv_norm + my_row);      // capacity is padded to whole tiles
#endif
                const uint4* base = p.rows + (size_t)row0 * PR + (size_t)g * PR + (RAGGED ? 0 : j);
                int acc[L];
#pragma unroll
                for (int r = 0; r < L; ++r) {
                    int a = 0;
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        // RAGGED: a lane slot beyond the row re-reads the row's last chunk against a zero query chunk:
                        // no branch, so the loads of an iteration stay batched
                        uint4 v = ldg_stream(base + (size_t)(r * G) * PR + (RAGGED ? coff[c] : (uint32_t)(c * L)));
                        a = dot16(v, q[c], a);
                    }
                    acc[r] = a;
                }
                const int s = transpose_reduce<L>(acc, j);
                const int dot_i = 2 * s + bias;
                const float kappa = __fmul_rn(__fmul_rn((float)dot_i, inv_r), qh.inv_q);
                if constexpr (!EXACT) {
                    const u64 key = make_key64(kappa, my_row);
#ifdef PBX_EXP_NOPUSH
                    if (key == 0x1234567ull) buf[0] = key;
#else
                    bool pass = my_row < p.n && key > tau && kappa_shift(kappa) >= gthr;
                    if constexpr (RESTRICT) {
                        const bool allowed = my_row < p.n && ((allow_word >> (my_row & 31u)) & 1u);
                        pass = pass && allowed && kappa <= cut;
                        n_above += __popc(__ballot_sync(0xFFFFFFFFu, allowed && kappa > cut));
                    }
                    tb.push_warp(pass, key);
                    if (pass) atomicAdd(p.hist + kappa_bin(kappa), 1u);
#ifdef PBX_EXP_PROFILE
                    if (pass) atomicAdd(&g_scan_prof[blockIdx.x][0], 1ull);
#endif
#endif
                } else {
                    bool pass = false;
                    KeyX key = KeyOps<KeyX>::lowest();
                    if (my_row < p.n && kappa >= theta && kappa <= cut && row_allowed(p.allow, my_row)) {
                        const ReplayOut ro = replay_row<false>(reinterpret_cast<const uint8_t*>(p.rows) + (size_t)my_row * ((size_t)PR * 16),
                                                               p.qbytes, p.q16, p.dim, qh.sum_cq, sh.lut);
                        float dist = ref_distance(qh.sa, ro.sb, ro.dot);
                        const int64_t id = __ldg(p.ids + my_row);
                        if (dist < p.max_dist && !page_before(p.cut, dist, id)) {
                            key = make_keyx(dist, id, my_row);
                            pass = keyx_gt(key, tau);
                        }
                    }
                    tb.push_warp(pass, key);
                }
                if constexpr (!EXACT) gb = max(gb, gb_new);
            }
            if constexpr (!EXACT) {
                if (warp == 0 && lane == 0 && gpoll > sh.gb) sh.gb = gpoll;
            }
            if constexpr (RESTRICT) {
                if (lane == 0 && n_above) atomicAdd(&p.cut->above, n_above);
            }
            continue;
        }
        // rendezvous: this warp is out of work, or the buffer needs cutting back
        if (!have && !counted) {
            counted = true;
            if (lane == 0) atomicAdd(&sh.done, 1u);
        }
#ifdef PBX_EXP_PROFILE
        const long long t_r0 = clock64();
#endif
        __syncthreads();
#ifdef PBX_EXP_PROFILE
        const long long t_r1 = clock64();
        if constexpr (!EXACT) PBX_PROF_ADD(2, t_r1 - t_r0);
#endif
        if (sh.done == (uint32_t)kScanWarps) break;          // uniform: done only changes before a rendezvous
        if constexpr (EXACT) tb.compact(); else block_select_top(tb, &sh.sel);
#ifdef PBX_EXP_PROFILE
        if constexpr (!EXACT) { PBX_PROF_ADD(3, clock64() - t_r1); PBX_PROF_ADD(1, 1); }
#endif
    }

    // final cut.  Fast pass: entries below the freshest global bin threshold go first (in place, one
    // barrier per 256 entries: survivors are written below the region already read), so the sort that
    // follows is over a handful of keys.
    if constexpr (!EXACT) {
        const float gfinal = bin_threshold(max(sh.gb, *reinterpret_cast<volatile uint32_t*>(gbin)));
        PBX_PROF_ADD(5, sh.cnt);
        tb.filter_inplace([gfinal](const u64& e) { return kappa_shift(key64_kappa(e)) >= gfinal; });
        if (sh.cnt > p.keep) block_select_top(tb, &sh.sel);      // uniform; only adversarial row orders get here
    }
    if constexpr (!EXACT) PBX_PROF_ADD(6, sh.cnt);
    tb.compact();
    const uint32_t c = sh.cnt < p.keep ? sh.cnt : p.keep;
    K* out = reinterpret_cast<K*>(p.cand);
    for (uint32_t i = threadIdx.x; i < c; i += blockDim.x) out[(size_t)i * gridDim.x + blockIdx.x] = buf[i];
    if (threadIdx.x == 0) p.cand_cnt[blockIdx.x] = c;
#ifdef PBX_EXP_PROFILE
    if constexpr (!EXACT) PBX_PROF_ADD(4, clock64() - t_kernel0);
#endif
}

// Any other pitch: one lane per row, query chunks from shared memory.  Correctness path for odd
// dims (the reference's BLOB column is length-agnostic, src/engine.rs:48); not tuned.
template <bool EXACT>
__global__ void __launch_bounds__(kScanThreads, 2)
scan_generic_kernel(const ScanParams p) {
    using K = typename std::conditional<EXACT, KeyX, u64>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    K* buf = reinterpret_cast<K*>(smem_raw);
    int4* sq = reinterpret_cast<int4*>(smem_raw + (size_t)p.cap * sizeof(K));   // [pitch16][2] int4
    __shared__ ScanShared<K, EXACT> sh;

    if constexpr (EXACT) {
        if (p.status->need_exact == 0) return;
        sh.lut[threadIdx.x & 255] = ref_decode(threadIdx.x & 255);
    }
    for (uint32_t i = threadIdx.x; i < p.pitch16 * 2; i += blockDim.x) sq[i] = __ldg(reinterpret_cast<const int4*>(p.q16) + i);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const QueryHeader qh = *p.qh;
    const int bias = -255 * qh.sum_cq;
    float theta = 0.0f;
    if constexpr (EXACT) theta = p.status->theta;
    const float cut = page_kappa_hi(p.cut);
    if (threadIdx.x == 0) { sh.cnt = 0; sh.tau = KeyOps<K>::lowest(); }
    TopBuf<K> tb{buf, &sh.cnt, &sh.tau, p.cap, p.keep};
    const uint32_t n_tiles = (p.n + kTileRows - 1) / kTileRows;

    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) sh.tile[0] = atomicAdd(p.tile_counter, 1u);
        if (sh.cnt + kTileRows > p.cap) tb.compact();
        __syncthreads();
        const uint32_t tile = sh.tile[0];
        if (tile >= n_tiles) break;
        const K tau = sh.tau;
        uint32_t n_above = 0;
        for (int it = 0; it < kItersPerTile; ++it) {
            const uint32_t my_row = tile * kTileRows + (uint32_t)(it * kScanWarps + warp) * kRowsPerWarpIter + lane;
            const float inv_r = __ldg(p.inv_norm + my_row);
            const uint4* rp = p.rows + (size_t)my_row * p.pitch16;
            int s = 0;
            for (uint32_t c = 0; c < p.pitch16; ++c) {
                uint4 v = __ldg(rp + c);
                int4 a = sq[2 * c], b = sq[2 * c + 1];
                int qq[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                s = dot16(v, qq, s);
            }
            const int dot_i = 2 * s + bias;
            const float kappa = __fmul_rn(__fmul_rn((float)dot_i, inv_r), qh.inv_q);
            if constexpr (!EXACT) {
                const u64 key = make_key64(kappa, my_row);
                const bool allowed = my_row < p.n && row_allowed(p.allow, my_row);
                const bool pass = allowed && key > tau && kappa <= cut;
                n_above += __popc(__ballot_sync(0xFFFFFFFFu, allowed && kappa > cut));
                tb.push_warp(pass, key);
                if (pass) atomicAdd(p.hist + kappa_bin(kappa), 1u);
            } else {
                bool pass = false;
                KeyX key = KeyOps<KeyX>::lowest();
                if (my_row < p.n && kappa >= theta && kappa <= cut && row_allowed(p.allow, my_row)) {
                    const ReplayOut ro = replay_row<false>(reinterpret_cast<const uint8_t*>(p.rows) + (size_t)my_row * ((size_t)p.pitch16 * 16),
                                                           p.qbytes, p.q16, p.dim, qh.sum_cq, sh.lut);
                    float dist = ref_distance(qh.sa, ro.sb, ro.dot);
                    const int64_t id = __ldg(p.ids + my_row);
                    if (dist < p.max_dist && !page_before(p.cut, dist, id)) {
                        key = make_keyx(dist, id, my_row);
                        pass = keyx_gt(key, tau);
                    }
                }
                tb.push_warp(pass, key);
            }
        }
        if constexpr (!EXACT) {
            if (lane == 0 && n_above) atomicAdd(&p.cut->above, n_above);
        }
    }
    tb.compact();
    const uint32_t c = sh.cnt < p.keep ? sh.cnt : p.keep;
    K* out = reinterpret_cast<K*>(p.cand);
    for (uint32_t i = threadIdx.x; i < c; i += blockDim.x) out[(size_t)i * gridDim.x + blockIdx.x] = buf[i];
    if (threadIdx.x == 0) p.cand_cnt[blockIdx.x] = c;
}

}  // namespace pbx

// Row pitches of 3, 5, 6 or 8 times a power of two (in 16-byte chunks): dims 48 ... 4096 such as 96, 192, 384, 768,
// 1536 (x3), 80, 160, 320, 640, 1280, 2560 (x5), 3072 (x6), 4096 (x8).  X(lanes per row, chunks per lane, CTAs per SM).
#define PBX_EXTRA_SHAPES(X)                                                                  \
    X(1, 3, 2) X(2, 3, 2) X(4, 3, 2) X(8, 3, 2) X(16, 3, 2) X(32, 3, 2)                      \
    X(1, 5, 2) X(2, 5, 2) X(4, 5, 2) X(8, 5, 2) X(16, 5, 2) X(32, 5, 2)                      \
    X(32, 6, 2) X(32, 8, 1)

// Every other pitch: the smallest of these (lanes, chunks, CTAs per SM) layouts that holds the row, run RAGGED.
#define PBX_RAGGED_SHAPES(X) X(8, 1, 4) X(16, 1, 2) X(32, 1, 2) X(32, 2, 2) X(32, 4, 2) X(32, 8, 1)
