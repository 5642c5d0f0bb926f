// batch.cuh -- kernel B: the batched-query path.  A batch of queries against the corpus is a dense
// s8 x u8 -> s32 contraction  S[q, r] = sum_i (q_i - 128) r_i,  run on the 5th-generation tensor cores
// (tcgen05.mma.kind::i8, accumulators in TMEM), with the top-k selection fused into the epilogue so the
// Q x N score matrix (10^10 entries for 1024 x 10M) never exists in memory.
//
//   operands       :  A = query bytes centred on 128, q' = q - 128 = q ^ 0x80 (s8), M = 128 queries per CTA and MMA;
//                     B = corpus bytes r (u8), N = 256 corpus rows per tile;  S = sum q' r
//   exact integers:  dot_i = sum c(q)c(r) = 4 S + (2 sum r - 255 d) + (-510 sum q')   (c(v) = 2v - 255)
//   ranking key   :  kappa' = fl(fl(dot_i) * inv_norm_r)      (the per-query factor 1/|c(q)| is applied later)
//
// Why queries are the M operand: an accumulator lane is then ONE query and its 32-bit columns are corpus rows, so an
// epilogue thread (one TMEM lane) holds 32 scores of the same query.  All of them share that query's threshold, and the
// 32 rows' norms / row terms enter only through their range (precomputed per 32-row block at load time): the whole
// selection test is  max(32 scores) >= one bound,  16 three-input integer max instructions per 32 scores instead of a
// compare per score.  (The first version had corpus rows on the lanes: a different bound per register, 5.4 issued
// instructions per score where the tensor pipe leaves room for 4.)
//
// Why N = 256: measured on this part (tools/umma_i8_peak.cu), a 128 x 128 x 32 i8 MMA takes 83 cycles instead of 64
// (6307 MACs/clk/SM), 128 x 192 and 128 x 256 run at the full 8192.  Why cta_group::2: with 256-row tiles one SM cannot
// hold both a whole batch of queries and two corpus tiles; a CTA pair splits the tile (128 rows each, fetched by the
// hardware from both shared memories) and holds 2 x 512 queries, so the corpus is streamed once per batch of 1024.
//
// Warp roles per CTA (576 threads): warp 16 streams corpus K-chunks (and the tile's row / block metadata) with TMA into
// mbarrier rings; warp 17 of the pair leader issues the MMAs into a ring of two TMEM accumulators (2 x 256 columns): its
// descriptors are ready before it waits for an accumulator, so that nothing but the issue itself follows the epilogue's
// last arrival; warps 0..15 are the epilogue: warp w owns TMEM lanes 32 (w % 4) .. +31 (queries) and a quarter of the
// columns (rows) of every accumulator, read 32 at a time.  Per 32 x 32 scores the common case is one tcgen05.ld, 16
// three-input maxima, one bound (select + FMA + add + conversion against per-query terms precomputed in shared memory)
// and one vote.  Survivors of the bound take the exact float test; the few that beat the threshold are staged per warp
// and pushed to the per-query candidate buffers.  Starting thresholds come from a seed pass of the same kernel over a
// strided sample of tiles (one bound per query and 32-row block, nothing pushed; batch_seed_select_kernel takes each
// query's keep-th largest); inside the main pass the thresholds tighten from per-query histograms of the accepted keys;
// batch_tighten_kernel cuts the buffers back to `keep` at the end.  The final candidates go through the same bit-exact
// re-rank and certificate as the single-query path (batch_finalize_kernel).
//
// What bounds the main pass (measured, profiles/README.md round 2c): with an epilogue that only loads the accumulators and
// hands them back a 128 x 256 stage still takes ~760 cycles at K = 64 (MMA: 256) and ~1380 at K = 256 (MMA: 1024) -- the
// hand-off is a latency chain (commit -> wait -> tcgen05.ld -> arrive -> wait -> issue -> MMA) and two accumulators are
// all the 512 TMEM columns hold.  The epilogue's own instructions come on top (IPC 0.4-0.6 per scheduler).
#pragma once
#include <cuda.h>
#include <cstdio>
#include <type_traits>
#include "rerank.cuh"

namespace pbx {

#ifndef PBX_BATCH_EPI_WARPS
#define PBX_BATCH_EPI_WARPS 16
#endif
constexpr int kBatchEpiWarps = PBX_BATCH_EPI_WARPS;   // 16: four per TMEM lane quarter, a quarter of an accumulator's columns each, read 32
                                                      // at a time (<= 96 registers); 8: two per quarter, 64 at a time (up to 168 registers).
                                                      // Measured at 10M x 256 x 1024: 2.44 ms with 16 warps, 2.64 ms with 8.
#ifndef PBX_BATCH_EPI_GROUPS
#define PBX_BATCH_EPI_GROUPS 1
#endif
// Epilogue warp groups: with G groups, group g drains the accumulator stages s = g (mod G) alone -- its warps read G times as
// many columns of G times fewer stages, the fixed cost per stage and warp is paid G times less often, and an accumulator
// goes back to the MMA thread when kBatchEpiWarps / G warps (not all of them) have read it.
constexpr int kBatchEpiGroups = PBX_BATCH_EPI_GROUPS;
constexpr int kBatchThreads = 64 + 32 * kBatchEpiWarps;   // epilogue warps, then the TMA producer warp, then the MMA issuer warp
// The two single-thread roles sit on the HIGHEST warp ids: the warp scheduler prefers high warp ids among eligible
// warps, and an MMA issuer that shares its scheduler with four polling epilogue warps of higher priority starves.
constexpr int kBatchTmaWarp = kBatchEpiWarps, kBatchMmaWarp = kBatchEpiWarps + 1;
constexpr int kBatchMaxStages = 8;           // corpus K-chunk ring depth (the host sizes it to the shared memory left)
constexpr uint32_t kBatchMaxQG = 512;        // resident queries per CTA
constexpr uint32_t kBatchCap = 4096;         // candidate buffer entries per query (small k)
constexpr uint32_t kBatchCapLarge = 16384;   // ... for keep > 512 (k = 1000 class)
constexpr uint32_t kBatchHistBins = 1024;    // per-query histogram of accepted keys over kappa in [-1, 1]
constexpr uint32_t kBatchStage = 32;         // staged candidates per epilogue warp

// ---- PTX helpers -------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// A value the compiler must keep in a register: without this it re-derives the address of a __shared__ object from
// SR_CgaCtaId (an S2UR with a long latency) at every use, also right behind a barrier wait on the hand-off's critical path.
__device__ __forceinline__ uint32_t keep_u32(uint32_t v) { uint32_t r; asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v)); return r; }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {        // shared::cluster address of `addr` in CTA `rank`
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// Arrive (+ expect_tx) on a barrier given by a shared::cluster address: the CTA's own barrier or its pair leader's.
// Default semantics (release at CTA scope) on purpose: a cluster-scope release compiles to MEMBAR.ALL.GPU, i.e. every
// arrive would wait for the thread's outstanding global stores and atomics (measured: 2.6 us per accumulator stage
// instead of 0.5).  What these arrives order is TMEM / shared-memory reuse, which the tcgen05 fences and the
// completed loads already guarantee.
__device__ __forceinline__ void mbar_expect_tx_at(uint32_t bar_addr, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cluster.b64 _, [%0], %1;" ::"r"(bar_addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_at(uint32_t bar_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}
// Spin on try_wait (which itself suspends the thread for a short, hardware-chosen time).  No suspend-time hint: with a
// long hint the waiter is parked in NANOSLEEP.SYNCS and, for barriers completed from the other CTA of a pair (multicast
// commits, remote arrives), was observed to wake up microseconds late -- 4.7 us per accumulator stage instead of 0.5.
// Always on a barrier of the executing CTA.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "PBX_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra PBX_DONE;\n\t"
        "bra PBX_WAIT;\n\t"
        "PBX_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// ... on a barrier given by its shared::cta address (hoisted out of the loops: the address of a __shared__ object is
// re-derived from the CTA's shared window at every use otherwise)
__device__ __forceinline__ void mbar_wait_at(uint32_t bar_addr, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "PBX_WAITA:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra PBX_DONEA;\n\t"
        "bra PBX_WAITA;\n\t"
        "PBX_DONEA:\n\t}" ::"r"(bar_addr), "r"(parity) : "memory");
}
// Pure polling (test_wait never suspends the thread): for the two accumulator hand-off waits when PBX_BATCH_SPIN is set
// (bit 0: the MMA thread's wait for the epilogue, bit 1: the epilogue's wait for the MMAs)
__device__ __forceinline__ void mbar_spin_at(uint32_t bar_addr, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "PBX_SPIN:\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra PBX_SPUN;\n\t"
        "bra PBX_SPIN;\n\t"
        "PBX_SPUN:\n\t}" ::"r"(bar_addr), "r"(parity) : "memory");
}
#ifndef PBX_BATCH_SPIN
#define PBX_BATCH_SPIN 0
#endif
#ifndef PBX_BATCH_LDPIPE       // experiment: second tcgen05.ld of a stage in flight while the first half is processed.  Measured
#define PBX_BATCH_LDPIPE 0     // slower (2.10 instead of 2.01 ms at 10M x 256, 2.69 instead of 2.47 ms at 12.5M x 64; 96 registers): off
#endif
template <int CG>
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint32_t bar_addr, int x, int y) {
    if constexpr (CG == 1)
        asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                     ::"r"(smem_u32(dst)), "l"(map), "r"(bar_addr), "r"(x), "r"(y) : "memory");
    else        // the completion may be signalled on the pair leader's barrier
        asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                     ::"r"(smem_u32(dst)), "l"(map), "r"(bar_addr), "r"(x), "r"(y) : "memory");
}
// L2 prefetch of one box of a tensor map: no shared memory, no barrier.  The ring in shared memory holds 4-5 tiles per SM
// (128-160 KB); a stream at HBM speed needs ~200 KB in flight per SM, the rest waits in L2.
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int x, int y) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(map), "r"(x), "r"(y) : "memory");
}
// plain (non-tensor) bulk copy global -> this CTA's shared memory, completing on one of its own barriers
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// K-major operand with a W-byte swizzle (W = 128, 64, 32: one K-chunk of W bytes per row, 8-row groups of 8 W bytes):
// start address >> 4, LBO unused (1), SBO = 8 W bytes, descriptor version 1, layout type 2 / 4 / 6.
__device__ __forceinline__ uint64_t umma_desc_k(const void* smem_ptr, uint32_t w) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_u32(smem_ptr) & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)((8u * w) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(w == 128 ? 2u : (w == 64 ? 4u : 6u)) << 61;
    return d;
}
template <int CG>
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    if constexpr (CG == 1)
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
            ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
    else
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
            ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
// Arrives on the barrier once every MMA issued so far by this thread has retired; cta_group::2: on the barrier at the
// same shared-memory offset in both CTAs of the pair.
template <int CG>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    if constexpr (CG == 1)
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
    else
        asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                     ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld64_issue(uint32_t taddr, uint32_t (&r)[64]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
        "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
        "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]), "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]),
          "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]), "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]),
          "=r"(r[46]), "=r"(r[47]), "=r"(r[48]), "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]),
          "=r"(r[55]), "=r"(r[56]), "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
        : "r"(taddr));
}
// The registers are operands of the wait, so that no use of them can be scheduled ahead of it.
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                   "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                   "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}
__device__ __forceinline__ void tmem_ld_wait64(uint32_t (&r)[64]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]),
                   "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]),
                   "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]),
                   "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31]), "+r"(r[32]), "+r"(r[33]), "+r"(r[34]), "+r"(r[35]), "+r"(r[36]),
                   "+r"(r[37]), "+r"(r[38]), "+r"(r[39]), "+r"(r[40]), "+r"(r[41]), "+r"(r[42]), "+r"(r[43]), "+r"(r[44]), "+r"(r[45]),
                   "+r"(r[46]), "+r"(r[47]), "+r"(r[48]), "+r"(r[49]), "+r"(r[50]), "+r"(r[51]), "+r"(r[52]), "+r"(r[53]), "+r"(r[54]),
                   "+r"(r[55]), "+r"(r[56]), "+r"(r[57]), "+r"(r[58]), "+r"(r[59]), "+r"(r[60]), "+r"(r[61]), "+r"(r[62]), "+r"(r[63])
                 :: "memory");
}
// overloads by register count
__device__ __forceinline__ void tmem_ld_issue(uint32_t taddr, uint32_t (&r)[32]) { tmem_ld32_issue(taddr, r); }
__device__ __forceinline__ void tmem_ld_issue(uint32_t taddr, uint32_t (&r)[64]) { tmem_ld64_issue(taddr, r); }
__device__ __forceinline__ void tmem_ld_done(uint32_t (&r)[32]) { tmem_ld_wait(r); }
__device__ __forceinline__ void tmem_ld_done(uint32_t (&r)[64]) { tmem_ld_wait64(r); }
__device__ __forceinline__ int max3(int a, int b, int c) { return max(max(a, b), c); }      // VIMNMX3 on sm_100

// ---- per-32-row block metadata (load time): what the epilogue's one-compare test needs from the rows --------------------
// blk[b] = { norm_lo, norm_hi, rowterm_max, rowterm_min (as int bits) } over rows [32 b, 32 b + 32) below n_rows:
// norm = 1 / inv_norm (f32 division, the same expression everywhere), rowterm = 2 sum r - 255 dim.
// One warp computes block b.
__device__ __forceinline__ void block_meta_warp(const float* __restrict__ inv_norm, const int* __restrict__ row_sum, uint32_t dim,
                                                uint64_t b, int lane, uint64_t n_rows, float4* __restrict__ blk) {
    const uint64_t row = b * 32 + (uint64_t)lane;
    const bool ok = row < n_rows;
    float inv_lo = ok ? inv_norm[row] : __int_as_float(0x7f800000), inv_hi = ok ? inv_norm[row] : 0.0f;
    int rt_max = ok ? 2 * row_sum[row] - 255 * (int)dim : INT_MIN;
    int rt_min = ok ? 2 * row_sum[row] - 255 * (int)dim : INT_MAX;
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        inv_lo = fminf(inv_lo, __shfl_xor_sync(0xFFFFFFFFu, inv_lo, off));
        inv_hi = fmaxf(inv_hi, __shfl_xor_sync(0xFFFFFFFFu, inv_hi, off));
        rt_max = max(rt_max, __shfl_xor_sync(0xFFFFFFFFu, rt_max, off));
        rt_min = min(rt_min, __shfl_xor_sync(0xFFFFFFFFu, rt_min, off));
    }
    if (lane == 0) {
        float4 m;
        m.x = inv_hi > 0.0f ? __fdiv_rn(1.0f, inv_hi) : 0.0f;          // smallest norm of the block
        m.y = inv_hi > 0.0f ? __fdiv_rn(1.0f, inv_lo) : 0.0f;          // largest
        m.z = 0.25f * (float)rt_max;                                   // exact: |rowterm| < 2^24 (the epilogue's bound subtracts it as is)
        m.w = __int_as_float(rt_min);
        blk[b] = m;
    }
}
__global__ void block_meta_kernel(const float* __restrict__ inv_norm, const int* __restrict__ row_sum, uint32_t dim,
                                  uint64_t first_block, uint64_t n_blocks, uint64_t n_rows, float4* __restrict__ blk) {
    const uint64_t b = first_block + (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= first_block + n_blocks) return;
    block_meta_warp(inv_norm, row_sum, dim, b, threadIdx.x & 31, n_rows, blk);
}

// ---- per-batch query preparation: one CTA per (padded) query ---------------------------------------------
struct BatchPrepParams {
    const uint8_t* queries;     // [nq][dim]
    uint32_t nq, dim, pitch;
    uint8_t* qpad;              // [nq_pad][pitch] query bytes ^ 0x80, zero padded (rows beyond nq are zero): the MMA's A operand
    int16_t* q16;               // [nq][pitch] centred (re-rank)
    uint8_t* qbytes;            // [nq][pitch]
    QueryHeader* qh;            // [nq]
    int* colterm;               // [nq_pad]  -510 * sum (q_i - 128)
    float* thr;                 // [nq_pad]  -inf for real queries, +inf for padding
    uint32_t* cand_cnt;         // [nq_pad]
    uint32_t* overflow;         // [nq_pad]
    uint32_t* bhist;            // [nq_pad][kBatchHistBins], zeroed here
    float* inv_q;               // [nq_pad]
};

__global__ void __launch_bounds__(128)
batch_prep_kernel(const BatchPrepParams p) {
    extern __shared__ __align__(16) float prep_sq[];       // [dim] squares of the decoded query (for the reference's norm fold)
    const uint32_t q = blockIdx.x;
    const bool real = q < p.nq;
    int s = 0, n2 = 0, raw = 0;
    for (uint32_t i = threadIdx.x; i < p.pitch; i += blockDim.x) {
        uint32_t v = 0;
        int c = 0;
        if (real && i < p.dim) { v = p.queries[(size_t)q * p.dim + i]; c = centre(v); }
        p.qpad[(size_t)q * p.pitch + i] = (real && i < p.dim) ? (uint8_t)(v ^ 0x80u) : (uint8_t)0;   // q - 128 as s8
        if (real) { p.q16[(size_t)q * p.pitch + i] = (int16_t)c; p.qbytes[(size_t)q * p.pitch + i] = (uint8_t)v; }
        if (real && i < p.dim) { const float a = ref_decode(v); prep_sq[i] = __fmul_rn(a, a); }
        s += c; n2 += c * c; raw += (int)v;
    }
    __shared__ int ss[32], sn[32], sr[32];
    for (int off = 16; off; off >>= 1) {
        s += __shfl_xor_sync(~0u, s, off); n2 += __shfl_xor_sync(~0u, n2, off); raw += __shfl_xor_sync(~0u, raw, off);
    }
    if ((threadIdx.x & 31) == 0) { ss[threadIdx.x >> 5] = s; sn[threadIdx.x >> 5] = n2; sr[threadIdx.x >> 5] = raw; }
    __syncthreads();
    if (threadIdx.x == 0) {
        int S = 0, N = 0, R = 0;
        for (uint32_t w = 0; w < (blockDim.x + 31) / 32; ++w) { S += ss[w]; N += sn[w]; R += sr[w]; }
        if (real) {
            // the query's own norm fold (src/engine.rs:580): strictly sequential f32 additions of the rounded squares
            float sa = 0.0f;
            for (uint32_t i = 0; i < p.dim; ++i) sa = __fadd_rn(sa, prep_sq[i]);
            QueryHeader h;
            h.sum_cq = S; h.norm2_q = N; h.inv_q = (float)(1.0 / sqrt((double)N)); h.sa = sa;
            p.qh[q] = h;
        }
        p.colterm[q] = -510 * (R - 128 * (int)p.dim);          // -510 * sum (q_i - 128)   (R = 0 for padding queries)
        p.thr[q] = real ? -__int_as_float(0x7f800000) : __int_as_float(0x7f800000);
        p.cand_cnt[q] = 0u;
        p.overflow[q] = 0;
        p.inv_q[q] = real ? (float)(1.0 / sqrt((double)N)) : 0.0f;
    }
    for (uint32_t i = threadIdx.x; i < kBatchHistBins; i += blockDim.x) p.bhist[(size_t)q * kBatchHistBins + i] = 0;
}

// The epilogue's bound, split so that one step costs a select, an FMA, an add and a conversion.  A score passes when
// fl(fl(dot_i) * inv_r) >= thr with dot_i = 4 S + rowterm + colterm.  With norm = 1 / inv_r inside [norm_lo, norm_hi] and
// rowterm <= rt_max over the 32 rows of a block, passing implies (in real numbers, up to the roundings of the test itself:
// relative 3 * 2^-24 of thr * norm)
//     S >= (thr * (thr >= 0 ? norm_lo : norm_hi) - colterm - rt_max) / 4.
// Evaluated as  v = floor(fma(t4, norm_sel, cq) - rq)  with
//     t4 = thr / 4, pushed 5e-6 (relative) towards -inf: covers the roundings of the exact test, of norm_lo / norm_hi (one
//          rounded division each) and of the product;
//     cq = -colterm / 4 - (1e-6 |colterm| + 8): colterm can exceed 2^24 (conversion error < 2^-24 |colterm|), the FMA and
//          the subtraction round once each at magnitudes below 2^26 (errors <= 4 each, in units of S / 4 ... <= 2 in v);
//     rq = rt_max / 4, exact in float (block metadata z).
// The float -> int conversion saturates, so the clamped +-1e30 thresholds become INT_MIN / INT_MAX.
__host__ __device__ inline float batch_bound_t4(const float thr) { return 0.25f * thr * (thr >= 0.0f ? 1.0f - 5.0e-6f : 1.0f + 5.0e-6f); }
__host__ __device__ inline float batch_bound_cq(const int ct) {
    const float c = (float)ct;
    return -0.25f * c - (1.0e-6f * fabsf(c) + 8.0f);
}

// ---- the contraction + selection kernel ---------------------------------------------------------------------
struct BatchMmaParams {
    CUtensorMap map_rows;       // corpus [capacity][pitch] u8, box {w bytes, tn / CG rows}, w-byte swizzle
    CUtensorMap map_q;          // padded queries [nq_pad][pitch] u8, box {w bytes, 256 or 128 rows (must divide qg)}
    const float* inv_norm;
    const int* row_sum;
    const float4* blk_meta;     // [capacity / 32]
    const int* colterm;         // [nq_pad]
    const float* thr;           // [nq_pad] starting thresholds on kappa' (MAIN)
    u64* cand;                  // [nq_pad][cap]
    uint32_t* cand_cnt;         // [nq_pad]
    uint32_t* overflow;         // [nq_pad]
    uint32_t* bhist;            // [nq_pad][kBatchHistBins] accepted keys per query and kappa bin (in-pass tightening)
    const float* inv_q;         // [nq_pad] 1 / |c(q)|  (0 for padding queries)
    float* thr_live;            // == thr, written: thresholds tightened while the pass runs
    float* seed_lb;             // SEED: [sample blocks][nq_pad] lower bounds of the best kappa' of each 32-row block
    const uint32_t* allow;      // filtered search: bit per row, NULL = every row.  Read from L2 on the seed and survivor
                                // paths only; the 32-row bound test of the main pass is unchanged (a looser bound is valid)
    PageCut* cut;               // paged search: [nq] cut and cursor per query, NULL = first pages.  Read on the seed and
                                // survivor paths only (kappa = kappa' * inv_q, the f32 product the finalize ranks by)
    uint32_t nq_pad;
    uint32_t keep;
    uint32_t cap;               // candidate buffer entries per query
    uint32_t n;                 // rows visible to this search
    uint32_t dim;
    uint32_t w;                 // K-chunk width in bytes = swizzle span: 128, 64 or 32
    uint32_t kc;                // K-chunks per row (pitch / w)
    uint32_t qg;                // queries resident per CTA: 128, 256, 384 or 512
    uint32_t groups;            // query groups of CG * qg queries; the grid holds a multiple of `groups` clusters
    uint32_t stages;            // corpus K-chunk ring depth
    uint32_t tn;                // corpus rows per tile = UMMA N (128 or 256)
    uint32_t n_tiles;           // tiles of this launch: tile index = tile_step * i, i < n_tiles
    uint32_t tile_step;         // 1: every tile (MAIN); > 1: a strided sample (SEED)
    uint32_t tile_base;         // first tile of this launch (MAIN passes over a long shard run in segments; 0 otherwise)
    uint32_t prefetch_tiles;    // tiles the producer prefetches into L2 ahead of the shared-memory ring (0: none)
    uint32_t exp_flags;         // experiment builds (PBX_BATCH_PROF) only
};

#ifdef PBX_BATCH_PROF
// experiment builds only: per-CTA cycle counters of the three roles
// [0] producer: wait a_empty  [1] producer: wait m_empty  [2] mma: wait acc_empty  [3] mma: wait a_full  [4] mma: total
// [5] epi warp 2: wait acc_full  [6] epi: ld  [7] epi: after arrive (process)  [8] epi: wait m_full  [9] epi total  [10] stages
__device__ unsigned long long g_batch_prof[2048][12];
#define PBX_BP_T() clock64()
#define PBX_BP_ADD(i, t0) bp_acc[(i) % 5] += (unsigned long long)(clock64() - (t0))       // register accumulators, written once per role
#else
#define PBX_BP_T() 0ll
#define PBX_BP_ADD(i, t0) do { (void)(t0); } while (0)
#endif
static_assert(true, "");
constexpr uint32_t kBatchMetaSlots = 4;      // (power of two) ring of per-tile metadata (inv_norm, row_sum, block metadata of the tile's rows)
constexpr uint32_t kBatchScrWords = 40;      // survivor scratch slot: 32 scores + {bound, threshold, colterm, query, first row, first column}
constexpr uint32_t kBatchScrSlots = 4;       // per epilogue warp: two for a deferred step, two for the step in hand

// Dynamic shared memory of batch_mma_kernel after the 1024-byte alignment fix-up; the host sizes the ring with it.
__host__ __device__ inline size_t batch_smem_fixed(uint32_t qg, uint32_t tn) {
    return (size_t)qg * 20                                            // s_colterm, s_thr, s_invq, s_t4, s_cq
           + (size_t)kBatchMetaSlots * (tn * 8 + tn / 2)              // metadata ring: inv_norm, row_sum, 16 B per 32 rows
           + (size_t)kBatchEpiWarps * kBatchScrSlots * kBatchScrWords * 4   // survivor scratch
           + (size_t)kBatchEpiWarps * kBatchStage * 12;               // staged candidates (key + query)
}

// SEED = true : thresholds do not exist yet.  Over a strided sample of tiles every (query, 32-row block) pair yields a
//               lower bound of the best kappa' in the block, from the block's maximal raw score and the block metadata;
//               batch_seed_select_kernel turns the `keep`-th largest bound of a query into its starting threshold (valid:
//               `keep` distinct rows are at least that good).  Same cost per score as the main pass, nothing is pushed.
// SEED = false: the main pass over all tiles with the selection described at the top of this file.
template <int CG, bool SEED>
__global__ void __launch_bounds__(kBatchThreads, 1)
batch_mma_kernel(const __grid_constant__ BatchMmaParams p) {
    extern __shared__ __align__(16) uint8_t bsm_raw[];     // NOT declared 1024-aligned: the compiler would fold the fix-up below away
    // the swizzle of TMA and UMMA is a function of the shared-memory address: tiles must sit on 1024-byte boundaries,
    // and dynamic shared memory only starts after the static variables (the host adds 1 KB of slack)
    uint8_t* bsm = bsm_raw + ((1024u - (smem_u32(bsm_raw) & 1023u)) & 1023u);
    constexpr uint32_t TN = 256u;                       // corpus rows per tile = UMMA N (p.tn agrees): at N = 128 the MMA runs at 77 % of the N = 256 rate
    constexpr uint32_t NB = TN / CG;                    // corpus rows of a tile in THIS CTA's shared memory: 128 per CTA of a pair, 256 for a single CTA
    constexpr uint32_t AS = 512u / TN;                  // TMEM accumulator ring: 2 x 256 or 4 x 128 columns
    constexpr uint32_t AS_LOG = AS == 2 ? 1u : 2u;
    constexpr uint32_t CPS = TN / 128u;                 // 32-column blocks per epilogue warp and accumulator
    const uint32_t QG = p.qg, KC = p.kc, W = p.w;
    const uint32_t MB = QG / 128u;                      // 128-query blocks = accumulator stages per tile
    const uint32_t STAGES = p.stages;
    const uint32_t stage_bytes = NB * W;
    uint8_t* sQ = bsm;                                  // [KC][QG][W]
    uint8_t* sA = bsm + (size_t)QG * KC * W;            // [STAGES][NB][W]
    float* s_minv = reinterpret_cast<float*>(sA + (size_t)STAGES * stage_bytes);   // [kBatchMetaSlots][TN] inv_norm of the tile's rows
    int* s_mrs = reinterpret_cast<int*>(s_minv + kBatchMetaSlots * TN);            // [kBatchMetaSlots][TN] row_sum
    float4* s_mblk = reinterpret_cast<float4*>(s_mrs + kBatchMetaSlots * TN);      // [kBatchMetaSlots][TN / 32] block metadata
    int* s_scr = reinterpret_cast<int*>(s_mblk + kBatchMetaSlots * (TN / 32u));    // [epilogue warp][kBatchScrSlots][kBatchScrWords] survivor scratch
    u64* st_key = reinterpret_cast<u64*>(s_scr + kBatchEpiWarps * kBatchScrSlots * kBatchScrWords);   // [epilogue warp][kBatchStage]
    uint32_t* st_q = reinterpret_cast<uint32_t*>(st_key + kBatchEpiWarps * kBatchStage);
    int* s_colterm = reinterpret_cast<int*>(st_q + kBatchEpiWarps * kBatchStage);
    float* s_thr = reinterpret_cast<float*>(s_colterm + QG);
    float* s_invq = s_thr + QG;
    float* s_t4 = s_invq + QG;          // threshold term of the epilogue's bound (batch_bound_t4)
    float* s_cq = s_t4 + QG;            // per-query constant of the bound (batch_bound_cq)
    __shared__ uint32_t st_cnt[kBatchEpiWarps];
    __shared__ __align__(8) uint64_t q_full, a_full[kBatchMaxStages], a_empty[kBatchMaxStages], acc_full[4], acc_empty[4];
    __shared__ __align__(8) uint64_t m_full[kBatchMetaSlots], m_empty[kBatchMetaSlots];
    __shared__ uint32_t tmem_base;

    // warp index through a shuffle: provably warp-uniform, so that the role loops below (executed by whole warps, one
    // elected lane issues) keep their descriptors and addresses in uniform registers; with per-thread values every
    // UTCIMMA / UTMALDG is wrapped in an ELECT + R2UR waterfall loop (measured: ~350 cycles per MMA issue instead of ~20)
    const int warp = __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
#ifdef PBX_BATCH_PROF
    unsigned long long bp_acc[5] = {0, 0, 0, 0, 0};
#endif
    const uint32_t rank = CG == 1 ? 0u : cluster_ctarank();
    const uint32_t cluster_id = blockIdx.x / CG;
    const uint32_t g = cluster_id % p.groups;                                   // query group of this cluster
    const uint32_t ci = cluster_id / p.groups, cstride = (gridDim.x / CG) / p.groups;
    const uint32_t qbase = (g * CG + rank) * QG;                                // first query of this CTA

    if (warp == kBatchMmaWarp) {
        if constexpr (CG == 1) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512u));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512u));
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
        }
    }
    if (threadIdx.x == 0) {
        // barriers that collect from both CTAs of a pair live in the leader and count CG arrivals
        mbar_init(&q_full, CG);
        for (int i = 0; i < kBatchMaxStages; ++i) { mbar_init(&a_full[i], CG); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < 4; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], CG * kBatchEpiWarps / kBatchEpiGroups); }
        for (uint32_t i = 0; i < kBatchMetaSlots; ++i) { mbar_init(&m_full[i], 1); mbar_init(&m_empty[i], kBatchEpiWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t i = threadIdx.x; i < QG; i += blockDim.x) {
        const int ct = p.colterm[qbase + i];
        const float th = fminf(fmaxf(p.thr[qbase + i], -1.0e30f), 1.0e30f);    // -inf: no bound known, +inf: padding query
        s_colterm[i] = ct;
        s_thr[i] = th;
        s_invq[i] = p.inv_q[qbase + i];
        s_t4[i] = batch_bound_t4(th);
        s_cq[i] = batch_bound_cq(ct);
    }
    if (threadIdx.x < kBatchEpiWarps) st_cnt[threadIdx.x] = 0;
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if constexpr (CG == 2) cluster_sync_all();          // the peer's barriers are initialised before anything signals them
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;

    if (warp == kBatchTmaWarp) {
        // ===== TMA producer (whole warp runs the loop, lane 0 issues): this CTA's queries (once), its NB rows of every
        // tile, and the tile's row / block metadata =====
        {
            const uint32_t qbox = (QG % 256u) ? 128u : 256u;       // rows per TMA box of the query operand: divides QG
            const uint32_t qfull_l = CG == 1 ? smem_u32(&q_full) : mapa_u32(smem_u32(&q_full), 0);
            if (lane == 0) mbar_expect_tx_at(qfull_l, QG * KC * W);
            for (uint32_t kc = 0; kc < KC; ++kc)
                for (uint32_t h = 0; h < QG; h += qbox)
                    if (lane == 0) tma_load_2d<CG>(sQ + ((size_t)kc * QG + h) * W, &p.map_q, qfull_l, (int)(kc * W), (int)(qbase + h));
            uint32_t st = 0, ph = 0, ti = 0;
            const uint32_t pf = p.prefetch_tiles;
            if (lane == 0)
                for (uint32_t d = 0; d < pf; ++d)
                    if (ci + d * cstride < p.n_tiles)
                        for (uint32_t kc = 0; kc < KC; ++kc)
                            tma_prefetch_2d(&p.map_rows, (int)(kc * W), (int)((p.tile_base + (ci + d * cstride) * p.tile_step) * TN + rank * NB));
            for (uint32_t i = ci; i < p.n_tiles; i += cstride, ++ti) {
                const uint32_t t = p.tile_base + i * p.tile_step;
                if (pf && lane == 0 && i + pf * cstride < p.n_tiles)
                    for (uint32_t kc = 0; kc < KC; ++kc)
                        tma_prefetch_2d(&p.map_rows, (int)(kc * W), (int)((p.tile_base + (i + pf * cstride) * p.tile_step) * TN + rank * NB));
                {
                    // inv_norm / row_sum / block metadata of the tile's TN rows (every CTA of a pair sees all of them):
                    // plain bulk copies into a small ring the epilogue reads in place
                    const uint32_t ms = ti & (kBatchMetaSlots - 1u);
                    const long long tp0 = PBX_BP_T();
                    mbar_wait(&m_empty[ms], ((ti >> 2) & 1u) ^ 1u);
                    PBX_BP_ADD(1, tp0);
                    if (lane == 0) {
                        mbar_expect_tx_at(smem_u32(&m_full[ms]), TN * 8u + (TN / 32u) * 16u);
                        bulk_load(s_minv + ms * TN, p.inv_norm + (size_t)t * TN, TN * 4u, &m_full[ms]);
                        bulk_load(s_mrs + ms * TN, p.row_sum + (size_t)t * TN, TN * 4u, &m_full[ms]);
                        bulk_load(s_mblk + ms * (TN / 32u), p.blk_meta + ((size_t)t * TN >> 5), (TN / 32u) * 16u, &m_full[ms]);
                    }
                }
                for (uint32_t kc = 0; kc < KC; ++kc) {
                    const long long tp1 = PBX_BP_T();
                    mbar_wait(&a_empty[st], ph ^ 1u);
                    PBX_BP_ADD(0, tp1);
                    const uint32_t full_l = CG == 1 ? smem_u32(&a_full[st]) : mapa_u32(smem_u32(&a_full[st]), 0);
                    if (lane == 0) {
#ifdef PBX_BATCH_PROF
                        if ((p.exp_flags & 1u) && ti >= 8u) {        // experiment: the MMAs run on stale tiles, nothing is streamed
                            mbar_arrive_at(full_l);
                        } else
#endif
                        {
                            mbar_expect_tx_at(full_l, stage_bytes);
                            tma_load_2d<CG>(sA + (size_t)st * stage_bytes, &p.map_rows, full_l, (int)(kc * W), (int)(t * TN + rank * NB));
                        }
                    }
                    if (++st == STAGES) { st = 0; ph ^= 1u; }
                }
            }
#ifdef PBX_BATCH_PROF
            if (lane == 0) { g_batch_prof[blockIdx.x][0] += bp_acc[0]; g_batch_prof[blockIdx.x][1] += bp_acc[1]; }
#endif
        }
    } else if (warp == kBatchMmaWarp) {
        // ===== MMA issuer (the whole warp of the pair leader runs the loop, lane 0 issues) =====
        if (rank == 0) {
            // instruction descriptor: D = s32 (2 << 4), A = s8 (1 at bit 7), B = u8 (0 at bit 10), both K-major,
            // N >> 3 at bit 17, M >> 4 at bit 24
            const uint32_t idesc = (2u << 4) | (1u << 7) | ((TN >> 3) << 17) | ((uint32_t)((128 * CG) >> 4) << 24);
            const uint32_t ksteps = W / 32u;
            mbar_wait(&q_full, 0);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t st0 = 0, ph0 = 0, acc_it = 0;
            const uint64_t da0 = umma_desc_k(sQ, W), db0 = umma_desc_k(sA, W);
            // Only the start-address field (the low word) of a descriptor changes from MMA to MMA, and everything the first
            // MMAs of a stage need is computed BEFORE the wait for the accumulator: between the epilogue's last arrival and
            // the first MMA lies nothing but the fence and the issue itself (the accumulator hand-off is a latency chain:
            // arrive -> wait -> issue -> MMA -> commit -> wait -> tcgen05.ld -> arrive, two of them in flight).
            const uint32_t da_lo = (uint32_t)da0, da_hi = (uint32_t)(da0 >> 32), db_lo = (uint32_t)db0, db_hi = (uint32_t)(db0 >> 32);
            const uint32_t a_kc = (QG * W) >> 4, a_mb = (128u * W) >> 4, b_st = stage_bytes >> 4;    // descriptor steps (16-byte units)
            const uint32_t acc_empty_l = keep_u32(smem_u32(&acc_empty[0])), a_full_l = keep_u32(smem_u32(&a_full[0]));
            const long long tm_all = PBX_BP_T();
            // one copy of the loop per K-chunk width: the MMAs of a chunk are then straight-line code with immediate offsets
            auto issue_all = [&](auto ks_c, auto kc_c) {
                constexpr uint32_t KS = decltype(ks_c)::value;          // MMAs (K = 32) per K-chunk = W / 32
                constexpr uint32_t KCC = decltype(kc_c)::value;         // K-chunks per row when known at compile time (0: p.kc)
                const uint32_t KCN = KCC ? KCC : KC;
                for (uint32_t i = ci; i < p.n_tiles; i += cstride) {
                    uint32_t st = st0, ph = ph0;
                    for (uint32_t mb = 0; mb < MB; ++mb, ++acc_it) {
                        const uint32_t ab = acc_it & (AS - 1u), par = (acc_it >> AS_LOG) & 1u;
                        const uint32_t d_tmem = tmem + ab * TN;
                        st = st0; ph = ph0;
                        uint32_t a_lo = da_lo + mb * a_mb, b_lo = db_lo + st * b_st;
                        uint64_t a_d = ((uint64_t)da_hi << 32) | (uint64_t)a_lo, b_d = ((uint64_t)db_hi << 32) | (uint64_t)b_lo;
                        asm volatile("" ::"l"(a_d), "l"(b_d), "r"(d_tmem), "r"(acc_empty_l + ab * 8u), "r"(idesc));
                        const long long tm0 = PBX_BP_T();
                        if (PBX_BATCH_SPIN & 1) mbar_spin_at(acc_empty_l + ab * 8u, par ^ 1u);
                        else mbar_wait_at(acc_empty_l + ab * 8u, par ^ 1u);           // the epilogues have drained its previous use
                        PBX_BP_ADD(2, tm0);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                        for (uint32_t kc = 0; kc < KCN; ++kc) {
                            if (mb == 0) {
                                const long long tm1 = PBX_BP_T();
                                mbar_wait_at(a_full_l + st * 8u, ph);
                                PBX_BP_ADD(3, tm1);
                                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                            }
                            if (lane == 0) {
                                const long long tm9 = PBX_BP_T();
    #pragma unroll
                                for (uint32_t ks = 0; ks < KS; ++ks)
                                    umma_i8<CG>(d_tmem, a_d + (uint64_t)(ks * 2u), b_d + (uint64_t)(ks * 2u), idesc, (kc | ks) ? 1u : 0u);
                                PBX_BP_ADD(0, tm9);
                                const long long tm10 = PBX_BP_T();
                                if (mb == MB - 1) umma_commit<CG>(&a_empty[st]);       // the stage is free once these MMAs retire
                                PBX_BP_ADD(1, tm10);
                            }
                            __syncwarp();
                            if (++st == STAGES) { st = 0; ph ^= 1u; }
                            a_lo += a_kc; b_lo = db_lo + st * b_st;
                            a_d = ((uint64_t)da_hi << 32) | (uint64_t)a_lo; b_d = ((uint64_t)db_hi << 32) | (uint64_t)b_lo;
                        }
                        if (lane == 0) umma_commit<CG>(&acc_full[ab]);
                        __syncwarp();
                    }
                    st0 = st; ph0 = ph;
                }
            };
            using std::integral_constant;
            if (ksteps == 4u && KC == 2u) issue_all(integral_constant<uint32_t, 4>{}, integral_constant<uint32_t, 2>{});         // dim 256
            else if (ksteps == 4u && KC == 1u) issue_all(integral_constant<uint32_t, 4>{}, integral_constant<uint32_t, 1>{});    // dim 128
            else if (ksteps == 2u && KC == 1u) issue_all(integral_constant<uint32_t, 2>{}, integral_constant<uint32_t, 1>{});    // dim 64
            else if (ksteps == 4u) issue_all(integral_constant<uint32_t, 4>{}, integral_constant<uint32_t, 0>{});
            else if (ksteps == 2u) issue_all(integral_constant<uint32_t, 2>{}, integral_constant<uint32_t, 0>{});
            else issue_all(integral_constant<uint32_t, 1>{}, integral_constant<uint32_t, 0>{});
            PBX_BP_ADD(4, tm_all);
#ifdef PBX_BATCH_PROF
            if (lane == 0) { g_batch_prof[blockIdx.x][2] += bp_acc[2]; g_batch_prof[blockIdx.x][3] += bp_acc[3]; g_batch_prof[blockIdx.x][4] += bp_acc[4];
                             g_batch_prof[blockIdx.x][11] += bp_acc[0]; g_batch_prof[blockIdx.x][10] += bp_acc[1] << 32; }
#endif
        }
    } else {
        // ===== epilogue: warp w owns TMEM lanes 32*(w%4) .. +31 (a hardware rule) = 32 queries of every 128-query block,
        // and columns [slice * TN/4, +TN/4) = corpus rows of the tile.  The MMA thread may run AS stages ahead.
        // Everything per-query or per-row is re-read from shared memory where it is used: the loop carries almost no
        // state besides the scores, because a spilled register costs an L2 round trip here (the L1 that would catch it
        // is the few KB the shared-memory carve-out leaves). =====
        const uint32_t e = (uint32_t)warp;
        const uint32_t quarter = (uint32_t)warp & 3u;
        constexpr uint32_t SLICES = kBatchEpiWarps / 4 / kBatchEpiGroups;  // warps that share a lane quarter of one accumulator
        const uint32_t slice = (e >> 2) % SLICES, group = (e >> 2) / SLICES;
        constexpr uint32_t cols_per_slice = TN / SLICES;                   // columns of this warp in every accumulator of its group
#ifndef PBX_BATCH_WIDTH
#define PBX_BATCH_WIDTH (kBatchEpiWarps == 8 ? 64u : 32u)
#endif
        constexpr uint32_t WIDTH = PBX_BATCH_WIDTH;                        // columns per tcgen05.ld (the live score registers)
        constexpr uint32_t STEPS = cols_per_slice / WIDTH;
        static_assert(cols_per_slice % WIDTH == 0 && STEPS >= 1, "epilogue column split");
        const uint32_t col_base = slice * cols_per_slice;
        uint32_t tile_iter = 0, acc_it = 0;
        const int dterm = -255 * (int)p.dim;
        u64* my_key = st_key + e * kBatchStage;
        uint32_t* my_q = st_q + e * kBatchStage;
        uint32_t* my_cnt = &st_cnt[e];
        int* my_scr = s_scr + e * (kBatchScrSlots * kBatchScrWords);   // survivor slots: 32 scores + {v, thr, ct, qi, row0, col0}
        const uint32_t acc_empty0 = keep_u32(CG == 1 ? smem_u32(&acc_empty[0]) : mapa_u32(smem_u32(&acc_empty[0]), 0));

        // Accepted candidates are staged per warp in shared memory and leave in two steps that never wait for each other
        // inside one accumulator stage: `flush_issue` sends the slot atomics of up to 32 staged records (their results stay
        // in registers, unread), `flush_complete`, one or more stages later, stores the keys to the slots that have arrived
        // by then.  A warp that waited ~2 us for its atomics right away would hold back the whole CTA pair: the MMA thread
        // needs every epilogue warp's arrival to reuse an accumulator.
        u64 pend_key = 0ull;
        uint32_t pend_q = 0, pend_slot = 0xFFFFFFFFu;                // 0xFFFFFFFF: nothing in flight
        auto hist_count = [&](u64 key, uint32_t qi) {                // every accepted key is counted once in its query's kappa histogram
            const float kap = __fmul_rn(key64_kappa(key), s_invq[qi - qbase]);
            const int bin = min(max(__float2int_rd(__fmul_rn(__fadd_rn(kap, 1.0f), (float)(kBatchHistBins / 2))), 0), (int)kBatchHistBins - 1);
            atomicAdd(p.bhist + (size_t)qi * kBatchHistBins + bin, 1u);
        };
        auto flush_complete = [&]() {
            if (pend_slot != 0xFFFFFFFFu) {
                if (pend_slot < p.cap) p.cand[(size_t)pend_q * p.cap + pend_slot] = pend_key;
                else p.overflow[pend_q] = 1u;
                pend_slot = 0xFFFFFFFFu;
            }
        };
        auto flush_issue = [&]() {                                   // warp-converged; nothing may be in flight
            __syncwarp();
            const uint32_t staged = min(*reinterpret_cast<volatile uint32_t*>(my_cnt), kBatchStage);
            if ((uint32_t)lane < staged) {
                pend_key = my_key[lane];
                pend_q = my_q[lane];
                pend_slot = min(atomicAdd(p.cand_cnt + pend_q, 1u), 0xFFFFFFFEu);
                hist_count(pend_key, pend_q);
            }
            __syncwarp();
            if (lane == 0) *my_cnt = 0;
            __syncwarp();
        };
        auto flush = [&]() { flush_complete(); flush_issue(); flush_complete(); };     // synchronous: refresh points, end of the pass
        // a record that does not fit the staging area (a burst of hits in one block): straight to global memory
        auto push_global = [&](u64 key, uint32_t qi) {
            const uint32_t slot = atomicAdd(p.cand_cnt + qi, 1u);
            if (slot < p.cap) p.cand[(size_t)qi * p.cap + slot] = key;
            else p.overflow[qi] = 1u;
            hist_count(key, qi);
        };
        // In-pass tightening.  At refresh points this CTA turns the histograms of the queries it is responsible for
        // (query j with j % clusters-in-group == its index) into thresholds -- the lower edge of the highest bin with at
        // least `keep` accepted keys at or above it, a valid bound because those keys are real rows -- publishes them
        // with an atomic max, and re-reads the published thresholds of all its queries.  One warp per histogram: the
        // 256 bins are one 16-byte load per lane pair, the suffix scan runs on shuffles.
        auto refresh = [&]() {
            flush();
            for (uint32_t j = ci % cstride + e * cstride; j < QG; j += kBatchEpiWarps * cstride) {     // warp-uniform
                const uint32_t qi = qbase + j;
                if (!(s_invq[j] > 0.0f)) continue;
                // lane l holds bins [l * PER, (l + 1) * PER): a suffix scan over lanes, then inside the crossing lane
                constexpr uint32_t PER = kBatchHistBins / 32u;
                const uint4* hp = reinterpret_cast<const uint4*>(p.bhist + (size_t)qi * kBatchHistBins + (size_t)lane * PER);
                uint32_t h[PER];
#pragma unroll
                for (uint32_t i4 = 0; i4 < PER / 4u; ++i4) {
                    const uint4 v4 = __ldcg(hp + i4);
                    h[4 * i4] = v4.x; h[4 * i4 + 1] = v4.y; h[4 * i4 + 2] = v4.z; h[4 * i4 + 3] = v4.w;
                }
                uint32_t mine = 0;
#pragma unroll
                for (uint32_t i = 0; i < PER; ++i) mine += h[i];
                uint32_t incl = mine;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const uint32_t x = __shfl_down_sync(0xFFFFFFFFu, incl, off);
                    if (lane + off < 32) incl += x;
                }
                const uint32_t above = incl - mine;                      // entries in higher bins than this lane's
                int bstar = -1;
                if (above < p.keep && above + mine >= p.keep) {
                    uint32_t run = above;
#pragma unroll
                    for (int i = (int)PER - 1; i >= 0; --i) { run += h[i]; if (bstar < 0 && run >= p.keep) bstar = lane * (int)PER + i; }
                }
                bstar = __reduce_max_sync(0xFFFFFFFFu, bstar);
                if (bstar > 0 && lane == 0) {
                    // kappa-bin edge back to kappa' units, nudged down so that no key of bin >= b* falls below it
                    const float edge = (float)bstar * (2.0f / (float)kBatchHistBins) - 1.0f;
                    float t = edge / s_invq[j];
                    t = t - fabsf(t) * 4.0e-6f - 1.0e-3f;
                    // float atomic max (thresholds may be negative): compare-and-swap on the bit pattern
                    float* addr = p.thr_live + qi;
                    float old = *reinterpret_cast<volatile float*>(addr);
                    while (t > old) {
                        const uint32_t prev = atomicCAS(reinterpret_cast<uint32_t*>(addr), __float_as_uint(old), __float_as_uint(t));
                        if (prev == __float_as_uint(old)) break;
                        old = __uint_as_float(prev);
                    }
                }
            }
            asm volatile("bar.sync 1, %0;" ::"r"(32 * kBatchEpiWarps) : "memory");       // the epilogue warps only
            for (uint32_t j = (uint32_t)threadIdx.x; j < QG; j += 32u * kBatchEpiWarps) {
                const float live = *reinterpret_cast<volatile float*>(p.thr_live + qbase + j);
                if (live > s_thr[j]) { s_thr[j] = fminf(live, 1.0e30f); s_t4[j] = batch_bound_t4(fminf(live, 1.0e30f)); }
            }
            asm volatile("bar.sync 1, %0;" ::"r"(32 * kBatchEpiWarps) : "memory");
        };

        // max of 32 scores: a tree of three-input maxima (16 instructions, depth 4)
        auto max32 = [](const uint32_t* r) {
            int t[11];
#pragma unroll
            for (int i = 0; i < 10; ++i) t[i] = max3((int)r[3 * i], (int)r[3 * i + 1], (int)r[3 * i + 2]);
            t[10] = max((int)r[30], (int)r[31]);
            const int u0 = max3(t[0], t[1], t[2]), u1 = max3(t[3], t[4], t[5]), u2 = max3(t[6], t[7], t[8]), u3 = max(t[9], t[10]);
            return max(max3(u0, u1, u2), u3);
        };
        // one bound per query and 32-row block: see batch_bound_t4 / batch_bound_cq
        auto bound = [](const float t4, const float cq, const float4 bm) {
            return __float2int_rd(fmaf(t4, t4 >= 0.0f ? bm.x : bm.y, cq) - bm.z);
        };
        // Rare: some lanes (queries) may have a hit among the 32 rows [row0, row0 + 32) whose scores they hold in r.  Such a
        // lane dumps its scores and {bound, threshold, colterm, query, first row, first column} into one of the warp's
        // scratch slots (`dump_lane`); the whole warp then tests one dumped query per step, one ROW per lane, against the
        // per-row metadata the producer left in shared memory (`test_slots`).  No unrolled per-register code, no register
        // carried across -- and a dump can be tested later, after the accumulator has been handed back.
        auto dump_lane = [&](const uint32_t* r, const int slot, const int v, const float thr, const int ct, const uint32_t qi,
                             const uint32_t row0, const uint32_t col0) {
            int* dst = my_scr + slot * kBatchScrWords;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                *reinterpret_cast<int4*>(dst + 4 * i) = make_int4((int)r[4 * i], (int)r[4 * i + 1], (int)r[4 * i + 2], (int)r[4 * i + 3]);
            *reinterpret_cast<int4*>(dst + 32) = make_int4(v, __float_as_int(thr), ct, (int)qi);
            *reinterpret_cast<int2*>(dst + 36) = make_int2((int)row0, (int)col0);
        };
        auto test_slots = [&](const int first, const int n_slots, const uint32_t ms) {      // warp-converged
            __syncwarp();
            for (int sl = first; sl < first + n_slots; ++sl) {
                const int* src = my_scr + sl * kBatchScrWords;
                const int4 h = *reinterpret_cast<const int4*>(src + 32);               // broadcast
                const int2 rc = *reinterpret_cast<const int2*>(src + 36);
                const int sc = src[lane];
                const uint32_t row = (uint32_t)rc.x + (uint32_t)lane;
                if (sc >= h.x && row < p.n && row_allowed(p.allow, row)) {
                    const uint32_t mi = ms * TN + (uint32_t)rc.y + (uint32_t)lane;
                    const int dot_i = 4 * sc + dterm + 2 * s_mrs[mi] + h.z;
                    const float kf = __fmul_rn((float)dot_i, s_minv[mi]);
                    // paged search: a row above the cut sorts before the cursor; it is counted, never pushed
                    const bool above = p.cut && __fmul_rn(kf, s_invq[(uint32_t)h.w - qbase]) > p.cut[h.w].kappa_hi;
                    if (above) atomicAdd(&p.cut[h.w].above, 1u);
                    else if (kf >= __int_as_float(h.y)) {
                        const u64 key = make_key64(kf, row);
                        const uint32_t slot = atomicAdd(my_cnt, 1u);
                        if (slot < kBatchStage) { my_key[slot] = key; my_q[slot] = (uint32_t)h.w; }
                        else push_global(key, (uint32_t)h.w);
                    }
                }
            }
            __syncwarp();
        };
        // dump + test right away, two lanes at a time (slots 2 and 3)
        auto resolve_now = [&](const uint32_t* r, uint32_t mask, const int v, const float thr, const int ct, const uint32_t qi,
                               const uint32_t row0, const uint32_t col0, const uint32_t ms) {
            while (mask) {
                const int o1 = __ffs(mask) - 1;
                mask &= mask - 1;
                const int o2 = mask ? __ffs(mask) - 1 : -1;
                mask &= mask - 1;                                        // (0 & anything) stays 0
                if (lane == o1 || lane == o2) dump_lane(r, lane == o2 ? 3 : 2, v, thr, ct, qi, row0, col0);
                test_slots(2, o2 >= 0 ? 2 : 1, ms);
            }
        };

#ifdef PBX_BATCH_PROF
        unsigned long long bp_stages = 0;
        auto g_prof_stage = [&]() { bp_stages += 1; };
        const long long te_all = clock64();
#else
        auto g_prof_stage = []() {};
#endif
        // 128-query blocks of this CTA in which this warp's lane quarter holds real queries (small batches: 8 queries occupy one
        // quarter of one block).  A quarter of padding queries has nothing to look at: it hands the accumulator straight back.
        uint32_t live_mb = 0;
        for (uint32_t mb = 0; mb < MB; ++mb)
            if (__any_sync(0xFFFFFFFFu, s_invq[mb * 128u + quarter * 32u + (uint32_t)lane] > 0.0f)) live_mb |= 1u << mb;
        const uint32_t acc_full0 = keep_u32(smem_u32(&acc_full[0])), m_full0 = keep_u32(smem_u32(&m_full[0])), m_empty0 = keep_u32(smem_u32(&m_empty[0]));
        for (uint32_t i = ci; i < p.n_tiles; i += cstride, ++tile_iter) {
            const uint32_t t = p.tile_base + i * p.tile_step;
            // refresh points: every tile at first (the starting thresholds are loose), then ever more rarely
            if (!SEED && tile_iter >= 1 && (tile_iter <= 8 || (tile_iter & (tile_iter - 1)) == 0 || (tile_iter & 31u) == 0)) refresh();
            const uint32_t ms = tile_iter & (kBatchMetaSlots - 1u);
            const long long te8 = PBX_BP_T();
            mbar_wait_at(m_full0 + ms * 8u, (tile_iter >> 2) & 1u);    // this tile's row / block metadata has landed
            if (threadIdx.x == 0) PBX_BP_ADD(8, te8);
            const float4* bmp = s_mblk + ms * (TN / 32u) + (col_base >> 5);
            for (uint32_t mb = 0; mb < MB; ++mb, ++acc_it) {
                if (kBatchEpiGroups > 1 && (acc_it % (uint32_t)kBatchEpiGroups) != group) continue;    // another group's stage
                const uint32_t ab = acc_it & (AS - 1u);
                const uint32_t j = mb * 128u + quarter * 32u + (uint32_t)lane;      // this lane's query in the block
                const float t4 = s_t4[j], cq = s_cq[j];
                const long long te5 = PBX_BP_T();
                if (PBX_BATCH_SPIN & 2) mbar_spin_at(acc_full0 + ab * 8u, (acc_it >> AS_LOG) & 1u);
                else mbar_wait_at(acc_full0 + ab * 8u, (acc_it >> AS_LOG) & 1u);
                if (threadIdx.x == 0) { PBX_BP_ADD(5, te5); g_prof_stage(); }
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t taddr = tmem + ((quarter * 32u) << 16) + ab * TN + col_base;
                if (!((live_mb >> mb) & 1u)) {
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive_at(acc_empty0 + ab * 8u);
                    continue;
                }
                // what is done with WIDTH scores of this lane's query (block(s) hf of the warp's column slice)
                auto process = [&](const uint32_t* r, const uint32_t hf) {
                    const float4 bm0 = bmp[hf * (WIDTH / 32u)];
                    const float4 bm1 = WIDTH == 64 ? bmp[hf * (WIDTH / 32u) + 1u] : bm0;
                    const int mx0 = max32(r), mx1 = WIDTH == 64 ? max32(r + WIDTH - 32) : mx0;
                    if constexpr (SEED) {
#ifdef PBX_BATCH_EXPSKIP      // timing experiments on the bare pass (PBX_BATCH_EXP=1: seed_lb == nullptr): 2 = max trees only, 3 = loads only
                        if (p.seed_lb == nullptr) {
                            if (PBX_BATCH_EXPSKIP == 2) { if (mx0 == 0x7FFFFFF1 || mx1 == 0x7FFFFFF1) p.overflow[0] = 1u; }
                            else { if (r[0] == 0x7FFFFFF1u && r[WIDTH - 1] == 0x7FFFFFF1u) p.overflow[0] = 1u; }
                            return;
                        }
#endif
                        // The block's best raw score belongs to a real row r* with dot_i = 4 S + rowterm + colterm >= 4 mx + rt_min
                        // + ct =: d and kappa' = fl(fl(dot_i) * inv_r), 1 / norm_hi <= inv_r <= 1 / norm_lo: kappa'(r*) >= d / norm_hi
                        // for d >= 0 and >= d / norm_lo otherwise (minus the roundings: relative 4e-6 and an absolute crumb).
                        const uint32_t col0 = col_base + WIDTH * hf;
                        const uint32_t qi = qbase + j;
                        const int ct = s_colterm[j];
                        const size_t blk = (size_t)((i * TN + col0) >> 5);
                        // Filtered or paged search: the bound of a block is that of its best ALLOWED row at or below the
                        // query's cut (the other columns do not count), -inf for a block without one.  The block's norm
                        // and rowterm range still brackets that row, so the bound stays valid, and `keep` finite bounds
                        // still stand for `keep` distinct searchable rows.
                        auto block_lb = [&](const uint32_t* rb, int mx, const float4 bm, const uint32_t row0, const uint32_t c0) {
                            if (p.allow || p.cut) {
                                uint32_t aw = p.allow ? __ldg(p.allow + (row0 >> 5)) : ~0u;       // the 32 rows of the block
                                if (p.cut && s_invq[j] > 0.0f) {               // (padding queries have no cut)
                                    const float hi = p.cut[qi].kappa_hi, iq = s_invq[j];
#pragma unroll
                                    for (int c = 0; c < 32; ++c) {
                                        const uint32_t mi = ms * TN + c0 + (uint32_t)c;
                                        const float kf = __fmul_rn((float)(4 * (int)rb[c] + dterm + 2 * s_mrs[mi] + ct), s_minv[mi]);
                                        if (__fmul_rn(kf, iq) > hi) aw &= ~(1u << c);
                                    }
                                }
                                if (aw == 0u) return -__int_as_float(0x7f800000);
                                int m = (int)0x80000000;
#pragma unroll
                                for (int c = 0; c < 32; ++c) m = ((aw >> c) & 1u) ? max(m, (int)rb[c]) : m;
                                mx = m;
                            }
                            const float d = (float)(4 * mx + __float_as_int(bm.w) + ct);
                            const float lb = d >= 0.0f ? __fdiv_rn(d, bm.y) : __fdiv_rn(d, bm.x);
                            return lb - fabsf(lb) * 4.0e-6f - 1.0e-3f;
                        };
                        const float lb0 = block_lb(r, mx0, bm0, t * TN + col0, col0);
                        if (p.seed_lb) p.seed_lb[blk * p.nq_pad + qi] = lb0;   // 32 queries per warp: one line
                        if constexpr (WIDTH == 64) {                      // (seed_lb is null only in the pipeline-rate experiment)
                            const float lb1 = block_lb(r + WIDTH - 32, mx1, bm1, t * TN + col0 + 32u, col0 + 32u);
                            if (p.seed_lb) p.seed_lb[(blk + 1) * p.nq_pad + qi] = lb1;
                        }
                    } else {
                        const int v0 = bound(t4, cq, bm0);
                        const uint32_t m0 = __ballot_sync(0xFFFFFFFFu, mx0 >= v0);
                        if (m0) {                                            // rare: fetch what only the survivor path needs
                            const uint32_t col0 = col_base + WIDTH * hf;
                            resolve_now(r, m0, v0, s_thr[j], s_colterm[j], qbase + j, t * TN + col0, col0, ms);
                        }
                        if constexpr (WIDTH == 64) {
                            const int v1 = bound(t4, cq, bm1);
                            const uint32_t m1 = __ballot_sync(0xFFFFFFFFu, mx1 >= v1);
                            if (m1) {
                                const uint32_t col0 = col_base + WIDTH * hf + 32u;
                                resolve_now(r + WIDTH - 32, m1, v1, s_thr[j], s_colterm[j], qbase + j, t * TN + col0, col0, ms);
                            }
                        }
                    }
                };
                auto hand_back = [&]() {                                 // the last scores are in registers: the MMA thread may reuse the accumulator
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive_at(acc_empty0 + ab * 8u);
                };
                const long long te6b = PBX_BP_T();
                if constexpr (STEPS == 2 && PBX_BATCH_LDPIPE) {
                    // the second load is in flight while the first 32 columns are looked at: only one tcgen05.ld round trip is
                    // exposed per stage, and the accumulator goes back before the second half is looked at
                    uint32_t ra[WIDTH], rb[WIDTH];
                    tmem_ld_issue(taddr, ra);
                    tmem_ld_done(ra);
                    tmem_ld_issue(taddr + WIDTH, rb);
                    process(ra, 0u);
                    tmem_ld_done(rb);
                    hand_back();
                    if (threadIdx.x == 0) PBX_BP_ADD(6, te6b);
                    process(rb, 1u);
                } else {
#pragma unroll
                    for (uint32_t hf = 0; hf < STEPS; ++hf) {          // WIDTH columns = one or two 32-row blocks at a time
                        uint32_t r[WIDTH];
                        tmem_ld_issue(taddr + WIDTH * hf, r);
                        tmem_ld_done(r);
                        if (hf == STEPS - 1) hand_back();
                        process(r, hf);
                    }
                }
            }
            if constexpr (!SEED) {
                // staged candidates: complete the flush issued a tile ago, issue the next one when enough are waiting
                __syncwarp();
                if (*reinterpret_cast<volatile uint32_t*>(my_cnt) >= kBatchStage / 2) { flush_complete(); flush_issue(); }
            }
            __syncwarp();                                            // done with this tile's metadata
            if (lane == 0) mbar_arrive_at(m_empty0 + ms * 8u);
        }
        if (!SEED) flush();
#ifdef PBX_BATCH_PROF
        if (threadIdx.x == 0) {
            g_batch_prof[blockIdx.x][9] += (unsigned long long)(clock64() - te_all);
            g_batch_prof[blockIdx.x][5] += bp_acc[0]; g_batch_prof[blockIdx.x][6] += bp_acc[1]; g_batch_prof[blockIdx.x][7] += bp_acc[2];
            g_batch_prof[blockIdx.x][8] += bp_acc[3]; g_batch_prof[blockIdx.x][10] += bp_stages;
        }
#endif
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if constexpr (CG == 2) cluster_sync_all();          // the pair's MMAs read both shared memories: leave together
    if (warp == kBatchMmaWarp) {
        if constexpr (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u));
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u));
    }
}

// ---- starting thresholds from the seed pass: thr[q] = the keep-th largest block bound of query q ---------------------
struct BatchSeedSelectParams {
    const float* seed_lb;       // [n_blocks][nq_pad]
    uint32_t n_blocks, nq_pad, keep;
    float* thr;                 // [nq_pad]
};

__global__ void __launch_bounds__(256)
batch_seed_select_kernel(const BatchSeedSelectParams p) {
    extern __shared__ __align__(16) unsigned char ssm[];
    u64* buf = reinterpret_cast<u64*>(ssm);              // [n_blocks] unique keys (ord(lb) << 32 | ~block)
    __shared__ uint32_t s_cnt;
    __shared__ u64 s_tau;
    __shared__ SelectScratch sel;
    const uint32_t q = blockIdx.x;
    if (p.n_blocks < p.keep) return;                     // fewer bounds than keep: no threshold (stays -inf)
    for (uint32_t i = threadIdx.x; i < p.n_blocks; i += blockDim.x) buf[i] = make_key64(__ldg(p.seed_lb + (size_t)i * p.nq_pad + q), i);
    if (threadIdx.x == 0) { s_cnt = p.n_blocks; s_tau = 0; }
    __syncthreads();
    if (p.n_blocks > p.keep) {
        TopBuf<u64> tb{buf, &s_cnt, &s_tau, p.n_blocks, p.keep};
        block_select_top(tb, &sel);
        if (threadIdx.x == 0) p.thr[q] = key64_kappa(s_tau);
    } else {
        __shared__ u64 s_min, s_scratch[32];
        block_min_key(buf, p.n_blocks, &s_min, s_scratch);
        if (threadIdx.x == 0) p.thr[q] = key64_kappa(s_min);
    }
}

// ---- between rounds: cut every query's candidate buffer back to `keep` and tighten its threshold ----------
struct BatchTightenParams {
    u64* cand;
    uint32_t* cand_cnt;
    float* thr;
    uint32_t keep;
    uint32_t nq;
    uint32_t cap;               // candidate buffer entries per query
};

__global__ void __launch_bounds__(256)
batch_tighten_kernel(const BatchTightenParams p) {
    extern __shared__ __align__(16) unsigned char tsm[];
    u64* buf = reinterpret_cast<u64*>(tsm);              // [cap]
    __shared__ uint32_t s_cnt;
    __shared__ u64 s_tau;
    __shared__ SelectScratch sel;
    const uint32_t q = blockIdx.x;
    const uint32_t c = min(p.cand_cnt[q], p.cap);
    if (c <= p.keep) return;                             // nothing to cut: the threshold stays where it is
    u64* src = p.cand + (size_t)q * p.cap;
    for (uint32_t i = threadIdx.x; i < c; i += blockDim.x) buf[i] = src[i];
    if (threadIdx.x == 0) { s_cnt = c; s_tau = 0; }
    __syncthreads();
    TopBuf<u64> tb{buf, &s_cnt, &s_tau, p.cap, p.keep};
    block_select_top(tb, &sel);
    const uint32_t kept = s_cnt;
    for (uint32_t i = threadIdx.x; i < kept; i += blockDim.x) src[i] = buf[i];
    if (threadIdx.x == 0) {
        p.cand_cnt[q] = kept;
        p.thr[q] = key64_kappa(s_tau);                   // every kept key has kappa' >= this
    }
}

// ---- the int8 tensor-pipe ceiling, measured (the denominator of the batched path's roofline) ---------------------------
// The batched kernel's MMA shape and nothing else: operands resident in shared memory (filled once, contents irrelevant),
// one thread per CTA pair issues tcgen05.mma.cta_group::2.kind::i8 (M = 256, N = 256, K = 256 bytes per accumulator) back
// to back into the ring of two TMEM accumulators; nobody reads them.  What is left is the tensor pipe and its
// shared-memory operand fetch.  pbx_int8_peak() times it; tools/umma_i8_peak.cu is the stand-alone form with more shapes.
__global__ void __launch_bounds__(128, 1)
batch_peak_kernel(int iters) {
    extern __shared__ __align__(16) uint8_t psm_raw[];
    uint8_t* psm = psm_raw + ((1024u - (smem_u32(psm_raw) & 1023u)) & 1023u);
    uint8_t* sa = psm;                                  // [2][128][128]
    uint8_t* sb = psm + 2 * 128 * 128;                  // [2][128][128]  (this CTA's half of the 256-row tile)
    __shared__ __align__(8) uint64_t bars[2];
    __shared__ uint32_t tmem_base;
    const int warp = __shfl_sync(0xFFFFFFFFu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
    for (uint32_t i = threadIdx.x; i < 4u * 128u * 128u / 4u; i += blockDim.x) reinterpret_cast<uint32_t*>(psm)[i] = 0x01020304u * (i | 1u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base)), "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = tmem_base;
    if (warp == 1 && cluster_ctarank() == 0) {
        const uint32_t idesc = (2u << 4) | (1u << 7) | ((256u >> 3) << 17) | ((256u >> 4) << 24);
        const uint64_t da0 = umma_desc_k(sa, 128), db0 = umma_desc_k(sb, 128);
        for (int it = 0; it < iters + 2; ++it) {
            const int s = it & 1;
            if (it >= 2) mbar_wait(&bars[s], ((it >> 1) - 1) & 1);
            if (it >= iters) continue;
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
#pragma unroll
                for (uint32_t kc = 0; kc < 2; ++kc)
#pragma unroll
                    for (uint32_t ks = 0; ks < 4; ++ks)
                        umma_i8<2>(tmem + s * 256u, da0 + (uint64_t)(kc * 1024u + ks * 2u), db0 + (uint64_t)(kc * 1024u + ks * 2u), idesc, (kc | ks) ? 1u : 0u);
                umma_commit<2>(&bars[s]);
            }
            __syncwarp();
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u));
}

// ---- batched finalize for keep <= 256: one small CTA per query, several per SM ----------------------------------------
// The same steps as finalize_kernel (candidate order, bit-exact replay, ORDER BY (dist, image_id), filter, LIMIT,
// certificate), sized for what a batched query leaves behind: at most `keep` candidates, one per thread (blockDim =
// keep rounded up to a warp).  Every thread replays its candidate row straight from global memory (the rows are random:
// no staging helps) against the decoded query in shared memory, with a byte -> float table replicated per lane
// (lut[v][lane]: one bank per lane, no conflicts whatever the bytes are); ranks are counted against shared memory with
// branch-free comparisons; the query's own norm fold comes from batch_prep_kernel (QueryHeader.sa).  1024 queries
// finish in two waves of small CTAs instead of seven waves of one 1024-thread CTA per SM.
constexpr uint32_t kBfThreads = 256;
struct BatchFinalizeParams {
    ExactLaunch x;              // exact-pass launch template (query 0); the launching CTA offsets the per-query pointers
    const u64* bcand;           // [nq][bcap] candidate keys (kappa' = dot_i * inv_norm_r, row)
    const uint32_t* bcnt;       // [nq]
    const uint32_t* boverflow;  // [nq]
    uint32_t* bticket;          // zero on entry and on exit
    uint32_t bcap, nq, keep, k, n, dim, pitch;
    const u64* n_allowed;       // filtered search: allowed rows among the n (device word), NULL = n
    const PageCut* cut;         // paged search: [nq] cut and cursor per query, NULL = first pages
    const uint8_t* rows;
    const int64_t* ids;
    const uint8_t* qbytes;      // [nq][pitch]
    const int16_t* q16;         // [nq][pitch]
    const QueryHeader* qh;      // [nq] (sa filled by batch_prep_kernel)
    double max_dist;
    float margin;
    pbx_hit* hits;              // [nq][k]
    uint32_t* count;            // [nq]
    SearchStatus* status;       // [nq]
};

// dynamic shared memory: decoded query [pitch] f32 | centred query [pitch] s16 | per-lane table [256][32] f32
__host__ __device__ inline size_t batch_finalize_smem(uint32_t pitch) { return (size_t)pitch * 6 + 256 * 32 * 4; }

__global__ void __launch_bounds__(kBfThreads, 3)
batch_finalize_kernel(const BatchFinalizeParams p) {
    extern __shared__ __align__(16) unsigned char bf_sm[];
    float* s_qa = reinterpret_cast<float*>(bf_sm);                                   // [pitch] decoded query (0 in the padding)
    int16_t* s_q16 = reinterpret_cast<int16_t*>(bf_sm + (size_t)p.pitch * 4);        // [pitch] centred query
    float* s_lut = reinterpret_cast<float*>(bf_sm + (size_t)p.pitch * 6);            // [256][32]
    __shared__ u64 s_key[kBfThreads];
    __shared__ uint32_t s_od[kBfThreads];
    __shared__ long long s_id[kBfThreads];
    __shared__ float s_kappa_k, s_kappa_last;
    __shared__ uint32_t s_pass, s_nonplateau, s_excl;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, q = blockIdx.x;
    const PageCut* cut_q = p.cut ? p.cut + q : nullptr;
    const uint32_t c = min(min(p.bcnt[q], p.bcap), blockDim.x);          // <= keep after the last batch_tighten
    const QueryHeader qh = p.qh[q];
    for (uint32_t i = tid; i < 256u * 32u; i += blockDim.x) s_lut[i] = ref_decode(i >> 5);
    for (uint32_t i = tid; i < p.pitch; i += blockDim.x) {
        s_qa[i] = i < p.dim ? ref_decode(p.qbytes[(size_t)q * p.pitch + i]) : 0.0f;
        s_q16[i] = p.q16[(size_t)q * p.pitch + i];
    }
    u64 key = 0ull;
    if (tid < c) {
        const u64 e = p.bcand[(size_t)q * p.bcap + tid];
        key = make_key64(__fmul_rn(key64_kappa(e), qh.inv_q), key64_row(e));
    }
    s_key[tid] = key;
    if (tid == 0) { s_kappa_k = 0.0f; s_kappa_last = 0.0f; s_pass = 0; s_nonplateau = 0; s_excl = 0; }
    __syncthreads();
    // candidate order by (kappa desc, row asc): what the certificate's two kappas are read from
    const uint32_t nc = min(c, p.keep);
    if (tid < c) {
        uint32_t rank = 0;
#pragma unroll 8
        for (uint32_t j = 0; j < c; ++j) rank += (s_key[j] > key) ? 1u : 0u;
        if (p.k > 0 && rank == p.k - 1 && nc >= p.k) s_kappa_k = key64_kappa(key);
        if (rank == nc - 1) s_kappa_last = key64_kappa(key);
        if (rank >= nc) key = 0ull;                                     // beyond keep (cannot happen after the tighten)
    }
    // kernel C: bit-exact replay of the reference distance for this thread's candidate (src/engine.rs:572-588): the two
    // f32 folds strictly in element order, the exact integer sums beside them
    float dist = __int_as_float(0x7f800000);
    int idot = 0, inorm = 0;
    long long id = INT64_MAX;
    bool have = tid < c && key != 0ull;
    if (have) {
        const uint32_t row = key64_row(key);
        const uint4* r4 = reinterpret_cast<const uint4*>(p.rows + (size_t)row * p.pitch);
        const float* lut = s_lut + lane;
        const uint32_t chunks = p.pitch >> 4, full = p.dim >> 4;
        float sb = 0.0f, fd = 0.0f;
        int acc = 0;
        unsigned s1 = 0, s2 = 0;
        uint4 cur = __ldg(r4), nxt = cur;
        for (uint32_t ch = 0; ch < chunks; ++ch) {
            if (ch + 1 < chunks) nxt = __ldg(r4 + ch + 1);
            const uint32_t w[4] = {cur.x, cur.y, cur.z, cur.w};
            if (ch < full) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 a = *reinterpret_cast<const float4*>(s_qa + 16 * ch + 4 * i);
                    const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const float fb = lut[((w[i] >> (8 * b)) & 255u) << 5];
                        sb = ref_fold(sb, fb, fb);
                        fd = ref_fold(fd, av[b], fb);
                    }
                }
            } else {                                            // ragged tail: dim is not a multiple of 16
                for (uint32_t i = 16 * ch; i < p.dim; ++i) {
                    const uint32_t o = i - 16 * ch;
                    const float fb = lut[((w[o >> 2] >> (8 * (o & 3))) & 255u) << 5];
                    sb = ref_fold(sb, fb, fb);
                    fd = ref_fold(fd, s_qa[i], fb);
                }
            }
            const int4 qa4 = *reinterpret_cast<const int4*>(s_q16 + 16 * ch), qb4 = *reinterpret_cast<const int4*>(s_q16 + 16 * ch + 8);
            const int qq[8] = {qa4.x, qa4.y, qa4.z, qa4.w, qb4.x, qb4.y, qb4.z, qb4.w};
            acc = dot16(cur, qq, acc);
            s1 = dp4a_uu(cur.x, 0x01010101u, s1); s1 = dp4a_uu(cur.y, 0x01010101u, s1);
            s1 = dp4a_uu(cur.z, 0x01010101u, s1); s1 = dp4a_uu(cur.w, 0x01010101u, s1);
            s2 = dp4a_uu(cur.x, cur.x, s2); s2 = dp4a_uu(cur.y, cur.y, s2);
            s2 = dp4a_uu(cur.z, cur.z, s2); s2 = dp4a_uu(cur.w, cur.w, s2);
            cur = nxt;
        }
        dist = ref_distance(qh.sa, sb, fd);
        idot = 2 * acc - 255 * qh.sum_cq;
        inorm = (int)(4u * s2 - 1020u * s1 + 65025u * p.dim);
        id = p.ids[row];
        if (page_before(cut_q, dist, id)) {
            // paged search: not on the page.  Taken out of the ranking (with its real dist it would sort first) and out
            // of the surviving candidates the certificate counts
            have = false;
            id = INT64_MAX;
            atomicAdd(&s_excl, 1u);
        }
    }
    const uint32_t od = have ? ord_f32(dist) : 0xFFFFFFFFu;
    s_od[tid] = od;
    s_id[tid] = id;
    __syncthreads();
    // ORDER BY dist ASC (ties by image_id), WHERE dist < ?, LIMIT k   (src/engine.rs:379-381).  Candidates are distinct
    // rows; equal (dist, id) pairs (duplicate ids in the table) fall back to the slot order.
    pbx_hit* hits_g = p.hits + (size_t)q * p.k;
    if (have) {
        uint32_t pos = 0;
#pragma unroll 4
        for (uint32_t j = 0; j < c; ++j) {
            const uint32_t oj = s_od[j];
            const long long ij = s_id[j];
            const bool before = (oj < od) | ((oj == od) & ((ij < id) | ((ij == id) & (j < tid))));
            pos += before ? 1u : 0u;
        }
        const bool ok = (double)dist < p.max_dist;
        if (ok) atomicAdd(&s_pass, 1u);
        if (dist < PBX_PLATEAU_DIST) atomicAdd(&s_nonplateau, 1u);
        if (pos < p.k) {
            pbx_hit hh;
            if (ok) { hh.image_id = id; hh.dist = dist; hh.dot = idot; hh.norm2 = inorm; hh.flags = 0; }
            else { hh.image_id = INT64_MAX; hh.dist = __int_as_float(0x7f800000); hh.dot = 0; hh.norm2 = 0; hh.flags = 0; }
            hits_g[pos] = hh;
        }
    }
    for (uint32_t i = nc - s_excl + tid; i < p.k; i += blockDim.x) {
        pbx_hit hh; hh.image_id = INT64_MAX; hh.dist = __int_as_float(0x7f800000); hh.dot = 0; hh.norm2 = 0; hh.flags = 0;
        hits_g[i] = hh;
    }
    if (s_excl) {
        // the certificate's kappa_k is that of the k-th best SURVIVING candidate (by kappa)
        __syncthreads();
        s_key[tid] = have ? key : 0ull;
        if (tid == 0) s_kappa_k = 0.0f;
        __syncthreads();
        if (have) {
            uint32_t rank = 0;
            for (uint32_t j = 0; j < c; ++j) rank += (s_key[j] > key) ? 1u : 0u;
            if (p.k > 0 && rank == p.k - 1) s_kappa_k = key64_kappa(key);
        }
    }
    __syncthreads();
    // certificate (DESIGN.md section 5), as in finalize_kernel
    if (tid == 0) {
        const uint32_t passing = s_pass;
        p.count[q] = passing < p.k ? passing : p.k;
        SearchStatus st;
        st.n_candidates = nc; st.reserved = 0; st.need_exact = 0; st.theta = 0.0f;
        u64 searchable = p.n_allowed ? *p.n_allowed : (u64)p.n;
        if (cut_q) searchable -= min(searchable, (u64)cut_q->above);     // paged search: rows at or below the cut
        if (searchable > nc) {
            const bool plateau_reachable = p.max_dist > (double)PBX_PLATEAU_DIST && s_nonplateau < p.k;
            const bool separated = (double)s_kappa_last < (double)s_kappa_k - (double)p.margin;
            const bool short_page = cut_q != nullptr && nc - s_excl < p.k;     // no k-th surviving candidate to bound with
            if (plateau_reachable || short_page) { st.need_exact = 1; st.theta = -__int_as_float(0x7f800000); }
            else if (!separated) { st.need_exact = 1; st.theta = (float)((double)s_kappa_k - (double)p.margin - 1e-7); }
        }
        if (p.boverflow[q] || p.bcnt[q] > blockDim.x) { st.need_exact = 1; st.theta = -__int_as_float(0x7f800000); }   // candidates were dropped
        p.status[q] = st;
        // the last CTA to finish tail-launches the exact pass of every query that needs one, one after the other
        // (they share the scan scratch), from a single thread so that their order is well defined.  bticket[1] counts
        // the queries that need one: normally zero, and then nobody walks the 1024 status words (a single thread
        // reading them one L2 round trip at a time was 250 us of the batch).
        if (st.need_exact) atomicAdd(p.bticket + 1, 1u);
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

}  // namespace pbx
