// api.cu -- the C ABI of include/pixelbox_b200.h: device-resident corpus shard, append, search.
// Host side of the hot path; the kernels are in scan.cuh / finalize.cuh.
#include <atomic>
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <type_traits>
#include <vector>

#include "finalize.cuh"
#include "batch.cuh"
#include "remove.cuh"
#include "replace.cuh"
#include "page.cuh"

using namespace pbx;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU_TRY(expr)                                                                               \
    do {                                                                                           \
        cudaError_t e__ = (expr);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return fail(e__ == cudaErrorMemoryAllocation ? PBX_E_OOM : PBX_E_CUDA, "%s failed: %s (%s:%d)", #expr, \
                        cudaGetErrorString(e__), __FILE__, __LINE__);                              \
    } while (0)

// ------------------------------------------------------------------------------------------------
// growable device arrays on CUDA virtual memory management
// ------------------------------------------------------------------------------------------------
// A shard's arrays grow by MAPPING more physical memory at the end of an address range reserved once (cuMemAddressReserve
// + cuMemCreate / cuMemMap on demand): the device pointers never move, nothing is copied, and a search that runs
// concurrently with the growth is not disturbed (the first version re-allocated x1.5, copied the whole shard device to
// device under the search lock and needed 2.5x the shard in HBM while doing so).  The driver entry points are fetched at
// run time (the library does not link libcuda); if they are missing, or PBX_NO_VMM is set, plain cudaMalloc + copy is used.
struct VmmApi {
    CUresult (*reserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
    CUresult (*free_)(CUdeviceptr, size_t) = nullptr;
    CUresult (*create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
    CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
    CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
    CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
    CUresult (*set_access)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
    CUresult (*granularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
    bool ok = false;
};
static const VmmApi& vmm_api() {
    static VmmApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        if (getenv("PBX_NO_VMM")) return;
        cudaDriverEntryPointQueryResult q;
        auto get = [&](const char* name, void** fn) { return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) == cudaSuccess && *fn != nullptr; };
        api.ok = get("cuMemAddressReserve", (void**)&api.reserve) && get("cuMemAddressFree", (void**)&api.free_) && get("cuMemCreate", (void**)&api.create) &&
                 get("cuMemRelease", (void**)&api.release) && get("cuMemMap", (void**)&api.map) && get("cuMemUnmap", (void**)&api.unmap) &&
                 get("cuMemSetAccess", (void**)&api.set_access) && get("cuMemGetAllocationGranularity", (void**)&api.granularity);
        cudaGetLastError();
    });
    return api;
}
struct VmmArray {
    CUdeviceptr base = 0;
    size_t reserved = 0, mapped = 0, gran = 0;
    std::vector<std::pair<CUmemGenericAllocationHandle, size_t>> chunks;
};
static CUmemAllocationProp vmm_prop(int device) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    return prop;
}
static bool vmm_reserve(VmmArray& a, int device, size_t bytes) {
    const VmmApi& api = vmm_api();
    const CUmemAllocationProp prop = vmm_prop(device);
    if (api.granularity(&a.gran, &prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED) != CUDA_SUCCESS || a.gran == 0) return false;
    a.reserved = (bytes + a.gran - 1) / a.gran * a.gran;
    return api.reserve(&a.base, a.reserved, 0, 0, 0) == CUDA_SUCCESS;
}
// Maps physical memory so that at least `need` bytes are backed.  Returns the newly mapped range in [*from, *to).
static int vmm_grow(VmmArray& a, int device, size_t need, size_t* from, size_t* to) {
    *from = *to = a.mapped;
    if (need <= a.mapped) return PBX_OK;
    if (need > a.reserved) return fail(PBX_E_CAPACITY, "shard outgrew the address range reserved for it (%zu > %zu bytes)", need, a.reserved);
    const VmmApi& api = vmm_api();
    const size_t add = (need - a.mapped + a.gran - 1) / a.gran * a.gran;
    const CUmemAllocationProp prop = vmm_prop(device);
    CUmemGenericAllocationHandle h;
    CUresult r = api.create(&h, add, &prop, 0);
    if (r != CUDA_SUCCESS) return fail(PBX_E_OOM, "cannot back %zu more bytes on device %d (cuMemCreate: %d)", add, device, (int)r);
    r = api.map(a.base + a.mapped, add, 0, h, 0);
    if (r == CUDA_SUCCESS) {
        CUmemAccessDesc acc = {};
        acc.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
        acc.location.id = device;
        acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        r = api.set_access(a.base + a.mapped, add, &acc, 1);
        if (r != CUDA_SUCCESS) api.unmap(a.base + a.mapped, add);
    }
    if (r != CUDA_SUCCESS) { api.release(h); return fail(PBX_E_CUDA, "mapping %zu bytes failed (%d)", add, (int)r); }
    a.chunks.emplace_back(h, add);
    *to = a.mapped + add;
    a.mapped += add;
    return PBX_OK;
}
static void vmm_release(VmmArray& a) {
    const VmmApi& api = vmm_api();
    if (a.base) {
        if (a.mapped) api.unmap(a.base, a.mapped);
        for (auto& c : a.chunks) api.release(c.first);
        api.free_(a.base, a.reserved);
    }
    a = VmmArray();
}

// ------------------------------------------------------------------------------------------------
// corpus
// ------------------------------------------------------------------------------------------------
struct pbx_corpus {
    int device = 0;
    int sm_count = 0;
    uint32_t dim = 0, pitch = 0, pitch16 = 0;
    std::atomic<uint64_t> n{0};       // committed rows (searches see a prefix)
    std::atomic<uint64_t> capacity{0};  // allocated (mapped) rows, multiple of kTileRows
    uint8_t* d_rows = nullptr;
    float* d_inv = nullptr;
    int* d_rsum = nullptr;            // sum of the raw bytes of each row (batched tensor-core path)
    float4* d_bmeta = nullptr;        // per 32-row block {norm_lo, norm_hi, rowterm_max}: the batched epilogue's bound
    bool use_vmm = false;             // the five arrays above live in reserved address ranges and grow by mapping (never move)
    VmmArray v_rows, v_inv, v_rsum, v_ids, v_bmeta;
    uint64_t reserved_rows = 0;       // rows the address ranges were reserved for
    // small appends are coalesced on the host and uploaded in blocks (or when a search needs them)
    std::vector<uint8_t> pend_rows;
    std::vector<int64_t> pend_ids;
    std::atomic<uint64_t> pending{0};
    int64_t* d_ids = nullptr;

    cudaStream_t stream = nullptr;    // default search stream
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_chain = nullptr;   // serialises searches enqueued on different streams
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    cudaEvent_t ev_s0 = nullptr, ev_s1 = nullptr;   // around the last fast-pass scan kernel of a timed search
    float last_scan_ms = 0.f;
    bool chain_valid = false;

    // per-batch query scratch
    uint32_t max_nq = 0;
    uint8_t* d_queries = nullptr;
    int16_t* d_q16 = nullptr;
    uint8_t* d_qbytes = nullptr;
    QueryHeader* d_qh = nullptr;
    SearchStatus* d_status = nullptr;
    unsigned char* d_split = nullptr;  // split finalize hand-over: keys[kMaxKeep] u64 | sbs, fdots, dots, norms [kMaxKeep] 4 B each | meta[4]
    bool split_finalize = true;        // PBX_NO_SPLIT_FINALIZE=1 keeps the one-kernel finalize for every shape
    size_t split_min_bytes = 256u * 1024u;   // keep * pitch from which the finalize is split (PBX_SPLIT_MIN_BYTES overrides)
    pbx_hit* d_hits = nullptr;
    size_t hits_cap = 0;
    // scan scratch
    void* d_cand = nullptr;
    size_t cand_bytes = 0;
    uint32_t* d_cand_cnt = nullptr;
    uint32_t* d_tile_counter = nullptr;
    uint32_t* d_hist = nullptr;       // kappa histogram of the scan CTAs' final lists (zeroed by the finalize kernel)
    unsigned long long* d_exact_passes = nullptr;
    // filtered searches (stream-ordered after ev_chain like the rest of the search scratch)
    uint32_t* d_allow = nullptr;      // bit per row: the row may be returned
    size_t allow_words = 0;
    u64* d_filter_words = nullptr;    // [0] allowed rows (mark_ids_kernel), [1] low word: a device filter was unsorted
    int64_t* d_filter_ids = nullptr;  // the sorted ids of a host-form filter
    size_t filter_ids_cap = 0;
    const uint32_t* cur_allow = nullptr;  // filter of the search being enqueued (NULL: none); exact_setup picks it up
    const u64* cur_allowed = nullptr;
    // paged searches (stream-ordered like the rest of the search scratch)
    PageCut* d_cut = nullptr;         // [cut_cap] cut and cursor per query (page_cut_kernel)
    pbx_hit* d_after = nullptr;       // [cut_cap] the cursors of a host-form call
    uint32_t cut_cap = 0;
    PageCut* cur_cut = nullptr;       // cuts of the search (or batch) being enqueued, one per query (NULL: first pages)
    // pinned staging
    uint8_t* h_queries = nullptr;
    size_t h_queries_cap = 0;
    pbx_hit* h_hits = nullptr;
    size_t h_hits_cap = 0;
    // zero-copy completion of single-query host calls: the kernels read the query from / write the hits to mapped pinned
    // memory and publish a sequence number the host polls (no copy engine, no stream synchronisation on the way)
    bool zero_copy = true;            // PBX_NO_ZEROCOPY=1: staged copies + cudaStreamSynchronize
    uint32_t* h_flag = nullptr;       // pinned, device-visible
    uint32_t flag_seq = 0;
    uint32_t* cur_done_flag = nullptr;   // what the kernels of the search being enqueued publish to (NULL: nothing)
    uint32_t cur_done_seq = 0;
    uint8_t* h_stage = nullptr;       // append staging: two slots of stage_rows rows + ids
    size_t h_stage_cap = 0, stage_rows = 0;
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};

    std::mutex mu;                    // searches and structural changes
    std::mutex append_mu;             // appends among themselves
    std::mutex grow_mu;               // growth steps among themselves (mapped growth runs outside append_mu)
    cudaStream_t grow_stream = nullptr;   // zero fill of freshly mapped memory

    uint32_t slack = 0;               // 0 = default
    uint32_t ctas_per_sm = 0;         // 0 = default
    uint64_t queries = 0;
    float last_search_ms = 0.f;
    uint64_t last_bytes = 0;
    int last_grid = 0;
    uint32_t last_n = 0;              // rows the last enqueued search saw
    uint64_t rows_generation = 0;     // bumped whenever the row buffers are re-allocated
    // batched (tensor-core) path
    uint32_t batch_pad = 0;           // padded queries the batch scratch is sized for
    uint8_t* d_qpad = nullptr;        // [batch_pad][pitch] raw query bytes, the MMA's B operand
    int* d_colterm = nullptr;
    float* d_thr = nullptr;
    uint32_t* d_bcnt = nullptr;
    uint32_t* d_boverflow = nullptr;
    u64* d_bcand = nullptr;           // [batch_pad][batch_cap]
    uint32_t batch_cap = 0;           // candidate buffer entries per query the scratch is sized for
    uint32_t* d_bhist = nullptr;      // [batch_pad][kBatchHistBins]
    float* d_binvq = nullptr;         // [batch_pad]
    float* d_seedlb = nullptr;        // [kBatchSeedTiles * 8][batch_pad] block bounds of the seed pass
    CUtensorMap map_rows, map_q;
    uint64_t map_rows_gen = ~0ull;
    uint32_t map_q_pad = 0, map_q_box = 0, map_rows_box = 0;
    uint32_t batch_cg = 0;            // CTAs per cluster of the batched kernel: 0 = by batch size; PBX_BATCH_CG=1 / 2 forces single CTAs / pairs

    uint32_t batch_min = 2;           // calls with at least this many queries use the tensor-core path
    uint64_t batched_queries = 0;
    bool scan_timed = false;          // ev_s0/ev_s1 were recorded by the last enqueue
    bool profiling = false;           // record CUDA events around the search / the scan (pbx_set_profiling)
};

constexpr size_t kStageMinRows = 2048;              // pinned upload staging: covers the coalesced blocks (kAppendBlock + kAppendCoalesceBelow rows)
static int ensure_stage(pbx_corpus* c, size_t rows_per_slot);

static uint32_t default_keep(uint32_t k, uint32_t slack) {
    uint32_t s = slack ? slack : std::max<uint32_t>(156u, k / 4u);
    uint32_t keep = k + s;
    if (!slack) keep = (keep + 31u) & ~31u;
    return std::min<uint32_t>(keep, kMaxKeep);
}

// Candidates per query of the batched path.  Its cost grows with keep (every candidate is a push from the tensor-core
// epilogue and the thresholds sit at the keep-th best), so the default slack is the smallest that keeps the certificate
// cheap to pass: max(28, k / 4) rows beyond k (keep = 128 for k = 100).  A certificate that fails -- ties or near-ties
// around rank k -- costs that query one exact pass, as in the single-query path.
static uint32_t batch_keep(uint32_t k, uint32_t slack) {
    if (slack) return std::min<uint32_t>(k + slack, kMaxKeep);
    const uint32_t keep = (k + std::max<uint32_t>(28u, k / 4u) + 31u) & ~31u;
    return std::min<uint32_t>(keep, kMaxKeep);
}

static float certificate_margin(uint32_t dim) {
    // 2 * (eps_d + 5u) + 2^-21 with eps_d = (2d + 1600) u, u = 2^-24   (DESIGN.md section 5)
    return (float)((4.0 * dim + 3232.0) * std::ldexp(1.0, -24));
}

static int free_corpus_buffers(pbx_corpus* c) {
    if (c->use_vmm) {
        vmm_release(c->v_rows); vmm_release(c->v_inv); vmm_release(c->v_rsum); vmm_release(c->v_ids); vmm_release(c->v_bmeta);
        c->d_rows = nullptr; c->d_inv = nullptr; c->d_ids = nullptr; c->d_rsum = nullptr; c->d_bmeta = nullptr;
        c->capacity = 0;
        c->use_vmm = false;
        return PBX_OK;
    }
    cudaFree(c->d_rows); cudaFree(c->d_inv); cudaFree(c->d_ids); cudaFree(c->d_rsum); cudaFree(c->d_bmeta);
    c->d_rows = nullptr; c->d_inv = nullptr; c->d_ids = nullptr; c->d_rsum = nullptr; c->d_bmeta = nullptr;
    c->capacity = 0;
    return PBX_OK;
}

// (re)allocates row storage for at least `rows` rows, keeping the committed prefix.  Caller holds mu.
// Growth on reserved address ranges: map more memory behind the arrays, zero it, done.  Pointers and committed rows stay
// where they are, so no search has to be kept out.  Caller holds grow_mu.
static int reserve_rows_vmm(pbx_corpus* c, uint64_t want) {
    struct Arr { VmmArray* a; size_t elem; } arrs[5] = {{&c->v_rows, (size_t)c->pitch}, {&c->v_inv, sizeof(float)}, {&c->v_rsum, sizeof(int)},
                                                        {&c->v_ids, sizeof(int64_t)}, {&c->v_bmeta, sizeof(float4)}};
    for (int i = 0; i < 5; ++i) {
        const size_t need = i == 4 ? (size_t)(want / 32) * arrs[i].elem : (size_t)want * arrs[i].elem;
        size_t from = 0, to = 0;
        int rc = vmm_grow(*arrs[i].a, c->device, need, &from, &to);
        if (rc != PBX_OK) return rc;
        // rows beyond the committed prefix are read (and ignored) by whole-tile loads: keep them defined
        if (to > from) CU_TRY(cudaMemsetAsync(reinterpret_cast<void*>(arrs[i].a->base + from), 0, to - from, c->grow_stream));
    }
    CU_TRY(cudaStreamSynchronize(c->grow_stream));
    c->capacity = want;
    return PBX_OK;
}

static int reserve_rows(pbx_corpus* c, uint64_t rows) {
    if (rows <= c->capacity) return PBX_OK;
    if (rows > PBX_MAX_ROWS) return fail(PBX_E_CAPACITY, "shard would hold %llu rows (max %llu)", (unsigned long long)rows, (unsigned long long)PBX_MAX_ROWS);
    // x1.5, and never less than 32 MB of rows per step once the shard exists: a growth step costs five driver mappings
    // plus a zero fill whatever its size, and an appender holds the append lock while it runs
    const uint64_t cap_now = c->capacity.load();
    uint64_t want = std::max<uint64_t>(rows, cap_now + cap_now / 2);
    if (cap_now) want = std::max<uint64_t>(want, cap_now + (32u << 20) / c->pitch);
    want = (want + kTileRows - 1) / kTileRows * kTileRows;
    if (c->use_vmm) {
        want = std::min<uint64_t>(want, c->reserved_rows);
        if (rows > c->reserved_rows) return fail(PBX_E_CAPACITY, "shard would hold %llu rows; its address range was reserved for %llu", (unsigned long long)rows, (unsigned long long)c->reserved_rows);
        int rc = reserve_rows_vmm(c, want);
        if (rc != PBX_OK && want > rows) {           // retry without growth head-room
            want = (rows + kTileRows - 1) / kTileRows * kTileRows;
            rc = reserve_rows_vmm(c, want);
        }
        return rc;
    }
    uint8_t* nr = nullptr; float* ni = nullptr; int64_t* nid = nullptr; int* ns = nullptr; float4* nb = nullptr;
    auto alloc_all = [&](uint64_t rows_) {
        cudaError_t e_ = cudaMalloc(&nr, rows_ * c->pitch);
        if (e_ == cudaSuccess) e_ = cudaMalloc(&ni, rows_ * sizeof(float));
        if (e_ == cudaSuccess) e_ = cudaMalloc(&nid, rows_ * sizeof(int64_t));
        if (e_ == cudaSuccess) e_ = cudaMalloc(&ns, rows_ * sizeof(int));
        if (e_ == cudaSuccess) e_ = cudaMalloc(&nb, rows_ / 32 * sizeof(float4));
        return e_;
    };
    auto free_all = [&]() {
        cudaFree(nr); cudaFree(ni); cudaFree(nid); cudaFree(ns); cudaFree(nb);
        nr = nullptr; ni = nullptr; nid = nullptr; ns = nullptr; nb = nullptr;
        cudaGetLastError();
    };
    cudaError_t e = alloc_all(want);
    if (e != cudaSuccess && want > rows) {          // retry without growth head-room
        free_all();
        want = (rows + kTileRows - 1) / kTileRows * kTileRows;
        e = alloc_all(want);
    }
    if (e != cudaSuccess) {
        free_all();
        return fail(PBX_E_OOM, "cannot allocate %llu rows x %u bytes on device %d: %s", (unsigned long long)want, c->pitch, c->device, cudaGetErrorString(e));
    }
    const uint64_t n = c->n.load();
    e = cudaDeviceSynchronize();                    // nothing may still read the old buffers
    if (e == cudaSuccess && n) {
        e = cudaMemcpyAsync(nr, c->d_rows, n * c->pitch, cudaMemcpyDeviceToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(ni, c->d_inv, n * sizeof(float), cudaMemcpyDeviceToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(nid, c->d_ids, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(ns, c->d_rsum, n * sizeof(int), cudaMemcpyDeviceToDevice, c->stream);
    }
    // block metadata: zero everywhere (a valid, merely loose bound), then the blocks of the committed rows again
    if (e == cudaSuccess) e = cudaMemsetAsync(nb, 0, want / 32 * sizeof(float4), c->stream);
    if (e == cudaSuccess && n) e = cudaMemcpyAsync(nb, c->d_bmeta, (n + 31) / 32 * sizeof(float4), cudaMemcpyDeviceToDevice, c->stream);
    // rows beyond the committed prefix are read (and ignored) by whole-tile loads: keep them defined
    if (e == cudaSuccess) e = cudaMemsetAsync(nr + n * c->pitch, 0, (want - n) * c->pitch, c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ni + n, 0, (want - n) * sizeof(float), c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(nid + n, 0, (want - n) * sizeof(int64_t), c->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(ns + n, 0, (want - n) * sizeof(int), c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) {                         // the old buffers stay in place, the new ones go
        free_all();
        return fail(PBX_E_CUDA, "moving %llu rows to the grown shard failed: %s", (unsigned long long)n, cudaGetErrorString(e));
    }
    cudaFree(c->d_rows); cudaFree(c->d_inv); cudaFree(c->d_ids); cudaFree(c->d_rsum); cudaFree(c->d_bmeta);
    c->d_rows = nr; c->d_inv = ni; c->d_ids = nid; c->d_rsum = ns; c->d_bmeta = nb;
    c->rows_generation++;                           // device pointers moved: tensor maps must be rebuilt
    c->capacity = want;
    return PBX_OK;
}

// Mapped growth (reserved address ranges) to at least `rows` rows; needs neither mu nor append_mu.
static int grow_mapped(pbx_corpus* c, uint64_t rows) {
    std::lock_guard<std::mutex> g(c->grow_mu);
    if (rows <= c->capacity.load()) return PBX_OK;
    CU_TRY(cudaSetDevice(c->device));
    return reserve_rows(c, rows);
}

static int ensure_query_scratch(pbx_corpus* c, uint32_t nq) {
    if (nq <= c->max_nq) return PBX_OK;
    CU_TRY(cudaDeviceSynchronize());
    cudaFree(c->d_queries); cudaFree(c->d_q16); cudaFree(c->d_qbytes); cudaFree(c->d_qh); cudaFree(c->d_status);
    c->d_queries = nullptr; c->d_q16 = nullptr; c->d_qbytes = nullptr; c->d_qh = nullptr; c->d_status = nullptr;
    c->max_nq = 0;
    uint32_t want = std::max<uint32_t>(nq, 64u);
    CU_TRY(cudaMalloc(&c->d_queries, (size_t)want * c->dim));
    CU_TRY(cudaMalloc(&c->d_q16, (size_t)want * c->pitch * sizeof(int16_t)));
    CU_TRY(cudaMalloc(&c->d_qbytes, (size_t)want * c->pitch));
    CU_TRY(cudaMalloc(&c->d_qh, (size_t)want * sizeof(QueryHeader)));
    CU_TRY(cudaMalloc(&c->d_status, (size_t)want * sizeof(SearchStatus)));
    if (!c->d_split) CU_TRY(cudaMalloc(&c->d_split, (size_t)kMaxKeep * 24 + 64));
    c->max_nq = want;
    return PBX_OK;
}

static int ensure_hits(pbx_corpus* c, size_t n_hits, uint32_t nq) {
    // [n_hits] records followed by [nq] counts, in units of records (24 bytes each)
    const size_t need = n_hits + ((size_t)nq * sizeof(uint32_t) + sizeof(pbx_hit) - 1) / sizeof(pbx_hit) + 1;
    if (need > c->hits_cap) {
        CU_TRY(cudaDeviceSynchronize());
        cudaFree(c->d_hits); c->d_hits = nullptr; c->hits_cap = 0;
        CU_TRY(cudaMalloc(&c->d_hits, need * sizeof(pbx_hit)));
        c->hits_cap = need;
    }
    if (need > c->h_hits_cap) {
        cudaFreeHost(c->h_hits);
        c->h_hits = nullptr; c->h_hits_cap = 0;
        CU_TRY(cudaMallocHost(&c->h_hits, need * sizeof(pbx_hit)));
        c->h_hits_cap = need;
    }
    return PBX_OK;
}

static int ensure_cand(pbx_corpus* c, size_t bytes) {
    if (bytes <= c->cand_bytes) return PBX_OK;
    CU_TRY(cudaDeviceSynchronize());
    cudaFree(c->d_cand); c->d_cand = nullptr; c->cand_bytes = 0;
    CU_TRY(cudaMalloc(&c->d_cand, bytes));
    c->cand_bytes = bytes;
    return PBX_OK;
}

// Row bitmap of filtered searches for `words` 32-row words, and room for `n_ids` host-form filter ids.
static int ensure_filter_scratch(pbx_corpus* c, size_t words, uint64_t n_ids) {
    if (!c->d_filter_words) CU_TRY(cudaMalloc(&c->d_filter_words, 2 * sizeof(u64)));
    if (words > c->allow_words) {
        words = std::max(words, c->allow_words + c->allow_words / 2);
        CU_TRY(cudaDeviceSynchronize());
        cudaFree(c->d_allow); c->d_allow = nullptr; c->allow_words = 0;
        CU_TRY(cudaMalloc(&c->d_allow, words * sizeof(uint32_t)));
        c->allow_words = words;
    }
    if (n_ids > c->filter_ids_cap) {
        const uint64_t want = std::max<uint64_t>(n_ids, c->filter_ids_cap + c->filter_ids_cap / 2);
        CU_TRY(cudaDeviceSynchronize());
        cudaFree(c->d_filter_ids); c->d_filter_ids = nullptr; c->filter_ids_cap = 0;
        CU_TRY(cudaMalloc(&c->d_filter_ids, want * sizeof(int64_t)));
        c->filter_ids_cap = want;
    }
    return PBX_OK;
}

// Cut and cursor of every query of a paged search, and room for the cursors of a host-form call.
static int ensure_page_scratch(pbx_corpus* c, uint32_t nq) {
    if (nq <= c->cut_cap) return PBX_OK;
    // + 1024: the batched kernels address the cuts of a 1024-query chunk by query slot, padding slots included
    const uint32_t want = std::max<uint32_t>(nq + 1024u, c->cut_cap + c->cut_cap / 2);
    CU_TRY(cudaDeviceSynchronize());
    cudaFree(c->d_cut); cudaFree(c->d_after); c->d_cut = nullptr; c->d_after = nullptr; c->cut_cap = 0;
    CU_TRY(cudaMalloc(&c->d_cut, (size_t)want * sizeof(PageCut)));
    CU_TRY(cudaMalloc(&c->d_after, (size_t)want * sizeof(pbx_hit)));
    c->cut_cap = want;
    return PBX_OK;
}

// Dynamic shared memory limits are per function and per device, and static shared memory counts
// against the 48 KB default as well: raise every kernel's cap once, when a corpus is created on a device.
template <typename Kern>
static cudaError_t allow_smem(Kern kern, size_t bytes) {
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}
constexpr uint64_t kBatchMaxRows = 0x7FFFF000ull;    // rows the batched path can address (TMA row coordinate is a signed 32-bit int)
constexpr uint32_t kBatchSegTilesLarge = 98304;      // main-pass segment (25M rows) between cut-backs when keep > 512
constexpr uint32_t kBatchSeedTiles = 256;            // sample tiles of the batched path's seed pass
constexpr size_t kBatchSmemLimit = 232448 - 1024;   // 227 KB per CTA minus the kernel's static shared memory
static cudaError_t init_kernel_attributes() {
    const size_t scan_cap = 8192 * sizeof(KeyX) + PBX_MAX_DIM * 2 + 1024;       // largest cap (keep 4096 + tile) + generic query stage
    const size_t fin_cap = 200 * 1024;
    cudaError_t e = cudaSuccess;
#define PBX_ALLOW(LL, CC)                                                                                       \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, false>, scan_cap);                                 \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, false, scan_minb(LL * CC), false, true>, scan_cap); \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, true>, scan_cap);
    PBX_ALLOW(1, 1) PBX_ALLOW(2, 1) PBX_ALLOW(4, 1) PBX_ALLOW(8, 1) PBX_ALLOW(16, 1) PBX_ALLOW(32, 1) PBX_ALLOW(32, 2) PBX_ALLOW(32, 4)
#undef PBX_ALLOW
#define PBX_ALLOW_M(LL, CC, MM)                                                                   \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, false, MM>, scan_cap);               \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, false, MM, false, true>, scan_cap);  \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, true, MM>, scan_cap);
    PBX_EXTRA_SHAPES(PBX_ALLOW_M)
#undef PBX_ALLOW_M
#define PBX_ALLOW_R(LL, CC, MM)                                                                  \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, false, MM, true>, scan_cap);        \
    if (e == cudaSuccess) e = allow_smem(scan_kernel<LL, CC, false, MM, true, true>, scan_cap);
    PBX_RAGGED_SHAPES(PBX_ALLOW_R)
#undef PBX_ALLOW_R
    if (e == cudaSuccess) e = allow_smem(scan_kernel<16, 1, false, 3>, scan_cap);
    if (e == cudaSuccess) e = allow_smem(scan_kernel<16, 1, false, 4>, scan_cap);
    if (e == cudaSuccess) e = allow_smem(scan_kernel<16, 1, false, 3, false, true>, scan_cap);
    if (e == cudaSuccess) e = allow_smem(scan_kernel<16, 1, false, 4, false, true>, scan_cap);
    if (e == cudaSuccess) e = allow_smem(scan_generic_kernel<false>, scan_cap);
    if (e == cudaSuccess) e = allow_smem(scan_generic_kernel<true>, scan_cap);
    if (e == cudaSuccess) e = allow_smem(prep_seed_kernel, PBX_MAX_DIM * 2 + 1024);
    if (e == cudaSuccess) e = allow_smem(finalize_kernel<false>, fin_cap);
    if (e == cudaSuccess) e = allow_smem(replay_kernel, (size_t)PBX_MAX_DIM * 6 + (size_t)kReplayRows * (kReplaySlice16 + 2) * 16);
    if (e == cudaSuccess) e = allow_smem(finalize_kernel<true>, fin_cap);
    if (e == cudaSuccess) e = allow_smem(batch_mma_kernel<1, false>, kBatchSmemLimit);
    if (e == cudaSuccess) e = allow_smem(batch_mma_kernel<1, true>, kBatchSmemLimit);
    if (e == cudaSuccess) e = allow_smem(batch_mma_kernel<2, false>, kBatchSmemLimit);
    if (e == cudaSuccess) e = allow_smem(batch_mma_kernel<2, true>, kBatchSmemLimit);
    if (e == cudaSuccess) e = allow_smem(batch_finalize_kernel, batch_finalize_smem(1024));
    if (e == cudaSuccess) e = allow_smem(batch_seed_select_kernel, (size_t)kBatchSeedTiles * 8u * sizeof(u64));
    if (e == cudaSuccess) e = allow_smem(batch_tighten_kernel, kBatchCapLarge * sizeof(u64));
    if (e == cudaSuccess) e = allow_smem(finalize_exact_kernel, fin_cap);
    return e;
}

extern "C" int pbx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

extern "C" const char* pbx_last_error(void) { return g_err; }
extern "C" const char* pbx_version(void) { return "pixelbox_b200 0.1.0 (sm_100a)"; }

extern "C" int pbx_corpus_create(uint32_t dim, uint64_t capacity_hint, int device, pbx_corpus** out) {
    if (!out) return fail(PBX_E_INVALID, "out is NULL");
    *out = nullptr;
    if (dim == 0 || dim > PBX_MAX_DIM) return fail(PBX_E_DIM, "dim %u outside [1, %u]", dim, PBX_MAX_DIM);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(PBX_E_NO_DEVICE, "no CUDA device visible: pixelbox_b200 has no CPU fallback");
    }
    if (device < 0 || device >= ndev) return fail(PBX_E_INVALID, "device %d out of range (have %d)", device, ndev);
    int major = 0, minor = 0;
    CU_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    CU_TRY(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
    if (major != 10) return fail(PBX_E_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, major, minor);
    CU_TRY(cudaSetDevice(device));
    pbx_corpus* c = new (std::nothrow) pbx_corpus();
    if (!c) return fail(PBX_E_OOM, "host allocation failed");
    c->device = device;
    c->dim = dim;
    c->split_finalize = getenv("PBX_NO_SPLIT_FINALIZE") == nullptr;
    if (const char* e = getenv("PBX_SPLIT_MIN_BYTES")) c->split_min_bytes = (size_t)atoll(e);
    c->zero_copy = getenv("PBX_NO_ZEROCOPY") == nullptr;
    if (const char* e = getenv("PBX_BATCH_CG")) c->batch_cg = atoi(e) == 1 ? 1u : (atoi(e) == 2 ? 2u : 0u);   // experiments
    c->pitch = (dim + 15u) & ~15u;
    c->pitch16 = c->pitch / 16u;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&c->grow_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_chain, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_t0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_t1);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_s0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev_s1);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_stage[0], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_stage[1], cudaEventDisableTiming);
    if (e == cudaSuccess) e = init_kernel_attributes();
    // Device-side (tail) launches of the exact pass: up to 2 per query of a 1024-query batch are queued by ONE finalize
    // grid.  The default pool holds 2048 pending launches; leave room for back-to-back batches.
    if (e == cudaSuccess) {
        size_t cur = 0;
        if (cudaDeviceGetLimit(&cur, cudaLimitDevRuntimePendingLaunchCount) == cudaSuccess && cur < 8192)
            e = cudaDeviceSetLimit(cudaLimitDevRuntimePendingLaunchCount, 8192);
    }
    if (e == cudaSuccess) e = cudaMallocHost(&c->h_flag, 64);
    if (e == cudaSuccess) *c->h_flag = 0;
    if (e == cudaSuccess) e = cudaMalloc(&c->d_cand_cnt, kMaxScanGrid * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&c->d_tile_counter, 512);      // [0] chunk counter, [32] global bin, +256 B exact-pass count
    if (e == cudaSuccess) e = cudaMemset(c->d_tile_counter, 0, 512);
    if (e == cudaSuccess) e = cudaMalloc(&c->d_hist, 2 * kHistBins * sizeof(uint32_t));     // scan histogram | seed histogram
    if (e == cudaSuccess) e = cudaMemset(c->d_hist, 0, 2 * kHistBins * sizeof(uint32_t));
    if (e == cudaSuccess) { c->d_exact_passes = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(c->d_tile_counter) + 256); }
    if (e != cudaSuccess) {
        int rc = fail(PBX_E_CUDA, "corpus setup failed: %s", cudaGetErrorString(e));
        pbx_corpus_destroy(c);
        return rc;
    }
    if (vmm_api().ok) {
        // address ranges for as many rows as the device could ever hold (HBM size / bytes per row), at most PBX_MAX_ROWS
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const uint64_t per_row = (uint64_t)c->pitch + 4 + 4 + 8 + 1;
        uint64_t max_rows = std::min<uint64_t>(PBX_MAX_ROWS, std::max<uint64_t>((uint64_t)total_b / per_row, capacity_hint) + kTileRows);
        max_rows = (max_rows + kTileRows - 1) / kTileRows * kTileRows;
        c->use_vmm = vmm_reserve(c->v_rows, device, max_rows * c->pitch) && vmm_reserve(c->v_inv, device, max_rows * sizeof(float)) &&
                     vmm_reserve(c->v_rsum, device, max_rows * sizeof(int)) && vmm_reserve(c->v_ids, device, max_rows * sizeof(int64_t)) &&
                     vmm_reserve(c->v_bmeta, device, max_rows / 32 * sizeof(float4));
        if (c->use_vmm) {
            c->reserved_rows = max_rows;
            c->d_rows = reinterpret_cast<uint8_t*>(c->v_rows.base); c->d_inv = reinterpret_cast<float*>(c->v_inv.base);
            c->d_rsum = reinterpret_cast<int*>(c->v_rsum.base); c->d_ids = reinterpret_cast<int64_t*>(c->v_ids.base);
            c->d_bmeta = reinterpret_cast<float4*>(c->v_bmeta.base);
        } else {
            vmm_release(c->v_rows); vmm_release(c->v_inv); vmm_release(c->v_rsum); vmm_release(c->v_ids); vmm_release(c->v_bmeta);
        }
    }
    {
        std::lock_guard<std::mutex> lk(c->mu);
        int rc = reserve_rows(c, std::max<uint64_t>(capacity_hint, 1));
        if (rc == PBX_OK) rc = ensure_stage(c, kStageMinRows);
        if (rc != PBX_OK) { pbx_corpus_destroy(c); return rc; }
    }
    *out = c;
    return PBX_OK;
}

extern "C" void pbx_corpus_destroy(pbx_corpus* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    free_corpus_buffers(c);
    cudaFree(c->d_queries); cudaFree(c->d_q16); cudaFree(c->d_qbytes); cudaFree(c->d_qh); cudaFree(c->d_status); cudaFree(c->d_split);
    cudaFree(c->d_qpad); cudaFree(c->d_colterm); cudaFree(c->d_thr); cudaFree(c->d_bcnt); cudaFree(c->d_boverflow); cudaFree(c->d_bcand);
    cudaFree(c->d_bhist); cudaFree(c->d_binvq); cudaFree(c->d_seedlb);
    cudaFree(c->d_hits); cudaFree(c->d_cand); cudaFree(c->d_cand_cnt); cudaFree(c->d_tile_counter); cudaFree(c->d_hist);
    cudaFree(c->d_allow); cudaFree(c->d_filter_words); cudaFree(c->d_filter_ids); cudaFree(c->d_cut); cudaFree(c->d_after);
    cudaFreeHost(c->h_queries); cudaFreeHost(c->h_hits); cudaFreeHost(c->h_stage); cudaFreeHost(c->h_flag);
    if (c->ev_chain) cudaEventDestroy(c->ev_chain);
    if (c->ev_t0) cudaEventDestroy(c->ev_t0);
    if (c->ev_t1) cudaEventDestroy(c->ev_t1);
    if (c->ev_s0) cudaEventDestroy(c->ev_s0);
    if (c->ev_s1) cudaEventDestroy(c->ev_s1);
    if (c->ev_stage[0]) cudaEventDestroy(c->ev_stage[0]);
    if (c->ev_stage[1]) cudaEventDestroy(c->ev_stage[1]);
    if (c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->grow_stream) cudaStreamDestroy(c->grow_stream);
    cudaGetLastError();
    delete c;
}

extern "C" int pbx_corpus_size(const pbx_corpus* c, uint64_t* n_rows) {
    if (!c || !n_rows) return fail(PBX_E_INVALID, "NULL argument");
    *n_rows = c->n.load() + c->pending.load(std::memory_order_acquire);      // pending (coalesced) appends are part of the table
    return PBX_OK;
}
extern "C" int pbx_corpus_synchronize(pbx_corpus* c) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    CU_TRY(cudaSetDevice(c->device));
    CU_TRY(cudaStreamSynchronize(c->stream));
    return PBX_OK;
}
extern "C" int pbx_corpus_dim(const pbx_corpus* c, uint32_t* dim) {
    if (!c || !dim) return fail(PBX_E_INVALID, "NULL argument");
    *dim = c->dim;
    return PBX_OK;
}

// Pinned staging of the uploads: two slots of rows_per_slot rows + ids.  Pinned allocations take milliseconds (and the
// searcher may be waiting for the append lock meanwhile): one at create sized for the coalesced blocks, larger ones only
// when a bulk load asks for them.
static int ensure_stage(pbx_corpus* c, size_t rows_per_slot) {
    const size_t per_row = (size_t)c->pitch + sizeof(int64_t);
    const size_t need = rows_per_slot * per_row * 2;
    if (c->h_stage_cap >= need) return PBX_OK;
    CU_TRY(cudaStreamSynchronize(c->copy_stream));
    cudaFreeHost(c->h_stage); c->h_stage = nullptr; c->h_stage_cap = 0; c->stage_rows = 0;
    CU_TRY(cudaMallocHost(&c->h_stage, need));
    c->h_stage_cap = need;
    c->stage_rows = rows_per_slot;
    return PBX_OK;
}

// copies n host rows to device rows [at, at+n) through pinned staging and computes their metadata
static int upload_rows(pbx_corpus* c, uint64_t at, const int64_t* ids, const uint8_t* hashes, uint64_t n) {
    const size_t max_stage_rows = std::max<size_t>(kStageMinRows, (size_t)(8u << 20) / c->pitch);
    const size_t per_row = (size_t)c->pitch + sizeof(int64_t);
    {
        size_t want = kStageMinRows;
        while (want < n && want < max_stage_rows) want *= 2;
        int rc0 = ensure_stage(c, std::min(want, max_stage_rows));
        if (rc0 != PBX_OK) return rc0;
    }
    const size_t stage_rows = c->stage_rows;
    cudaEvent_t* done = c->ev_stage;
    int rc = PBX_OK;
    uint64_t off = 0;
    int slot = 0;
    bool used[2] = {false, false};
    while (off < n && rc == PBX_OK) {
        const uint64_t m = std::min<uint64_t>(stage_rows, n - off);
        uint8_t* hs = c->h_stage + (size_t)slot * stage_rows * per_row;
        int64_t* hid = reinterpret_cast<int64_t*>(hs + stage_rows * c->pitch);
        if (used[slot]) cudaEventSynchronize(done[slot]);
        if (c->pitch == c->dim) {
            memcpy(hs, hashes + off * c->dim, m * c->dim);
        } else {
            memset(hs, 0, m * c->pitch);
            for (uint64_t r = 0; r < m; ++r) memcpy(hs + r * c->pitch, hashes + (off + r) * c->dim, c->dim);
        }
        memcpy(hid, ids + off, m * sizeof(int64_t));
        cudaError_t e = cudaMemcpyAsync(c->d_rows + (at + off) * c->pitch, hs, m * c->pitch, cudaMemcpyHostToDevice, c->copy_stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_ids + at + off, hid, m * sizeof(int64_t), cudaMemcpyHostToDevice, c->copy_stream);
        if (e == cudaSuccess) {
            const unsigned warps_per_block = 8;
            const unsigned blocks = (unsigned)((m + warps_per_block - 1) / warps_per_block);
            row_meta_kernel<<<blocks, warps_per_block * 32, 0, c->copy_stream>>>(reinterpret_cast<const uint4*>(c->d_rows), c->pitch16, c->dim,
                                                                                at + off, m, c->d_inv, c->d_rsum);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaEventRecord(done[slot], c->copy_stream);
        if (e != cudaSuccess) rc = fail(PBX_E_CUDA, "row upload failed: %s", cudaGetErrorString(e));
        used[slot] = true;
        slot ^= 1;
        off += m;
    }
    if (rc == PBX_OK && n) {
        // per-32-row block metadata of every block that holds one of the new rows (the first one may be shared with
        // committed rows: its bound can only widen, which a concurrent search tolerates)
        const uint64_t b0 = at / 32, b1 = (at + n + 31) / 32;
        block_meta_kernel<<<(unsigned)((b1 - b0 + 7) / 8), 256, 0, c->copy_stream>>>(c->d_inv, c->d_rsum, c->dim, b0, b1 - b0, at + n, c->d_bmeta);
        if (cudaGetLastError() != cudaSuccess) rc = fail(PBX_E_CUDA, "block metadata launch failed");
    }
    cudaError_t e = cudaStreamSynchronize(c->copy_stream);
    if (rc == PBX_OK && e != cudaSuccess) rc = fail(PBX_E_CUDA, "row upload failed: %s", cudaGetErrorString(e));
    return rc;
}

// Caller holds append_mu.
static int append_locked(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n) {
    CU_TRY(cudaSetDevice(c->device));
    const uint64_t at = c->n.load();
    if (at + n > c->capacity) {
        int rc;
        if (c->use_vmm) {
            rc = grow_mapped(c, at + n);                // maps more memory behind the arrays: searches keep running
        } else {
            std::lock_guard<std::mutex> lk(c->mu);      // growth moves the buffers: no search may be running
            rc = reserve_rows(c, at + n);
        }
        if (rc != PBX_OK) return rc;
    }
    // rows beyond the committed prefix are invisible to concurrent searches until n is published
    int rc = upload_rows(c, at, image_ids, hashes, n);
    if (rc != PBX_OK) return rc;
    c->n.store(at + n);
    return PBX_OK;
}

// Small appends (the indexer inserts one image at a time, src/engine.rs:186-203) are collected on the host and uploaded
// in blocks: one staged copy + metadata launch + synchronisation per kAppendBlock rows instead of per row.  Pending rows
// are part of the table: the size includes them and every search uploads them first.  Caller holds append_mu.
constexpr uint64_t kAppendCoalesceBelow = 64;       // appends of fewer rows than this are collected
constexpr uint64_t kAppendBlock = 1024;             // ... and uploaded when this many are waiting
static int flush_pending_locked(pbx_corpus* c) {
    const uint64_t m = c->pend_ids.size();
    if (m == 0) return PBX_OK;
    int rc = append_locked(c, c->pend_ids.data(), c->pend_rows.data(), m);
    if (rc != PBX_OK) return rc;                    // the rows stay pending
    c->pend_ids.clear();
    c->pend_rows.clear();
    c->pending.store(0, std::memory_order_release);
    return PBX_OK;
}
static int flush_pending(pbx_corpus* c) {
    if (c->pending.load(std::memory_order_acquire) == 0) return PBX_OK;
    std::lock_guard<std::mutex> alk(c->append_mu);
    return flush_pending_locked(c);
}

extern "C" int pbx_corpus_append(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (n == 0) return PBX_OK;
    if (!image_ids || !hashes) return fail(PBX_E_INVALID, "NULL ids or hashes with n > 0");
    if (c->use_vmm) {
        // Grow AHEAD of need and outside the append lock: a searcher that has to flush pending rows waits for that lock,
        // and a growth step (five driver mappings + a zero fill) takes about a millisecond.  Failure here is not an error
        // yet: the rows may still fit, and append_locked reports it if they do not.
        const uint64_t soon = c->n.load() + c->pending.load(std::memory_order_acquire) + n + 4 * kAppendBlock;
        if (soon > c->capacity.load() && soon <= c->reserved_rows) { if (grow_mapped(c, soon) != PBX_OK) g_err[0] = 0; }
    }
    std::lock_guard<std::mutex> alk(c->append_mu);
    if (n < kAppendCoalesceBelow) {
        try {
            c->pend_ids.insert(c->pend_ids.end(), image_ids, image_ids + n);
            c->pend_rows.insert(c->pend_rows.end(), hashes, hashes + n * c->dim);
        } catch (...) { return fail(PBX_E_OOM, "host allocation failed"); }
        c->pending.store(c->pend_ids.size(), std::memory_order_release);
        return c->pend_ids.size() >= kAppendBlock ? flush_pending_locked(c) : PBX_OK;
    }
    int rc = flush_pending_locked(c);               // keep the order of arrival
    if (rc != PBX_OK) return rc;
    return append_locked(c, image_ids, hashes, n);
}

extern "C" int pbx_corpus_flush(pbx_corpus* c) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    return flush_pending(c);
}

// Rows that are already on the device (embeddings quantized there): [n][dim] bytes and [n] ids, both DEVICE pointers on
// the corpus' device.  Copies them behind the committed rows on `cuda_stream`, computes their metadata, waits for that
// stream and publishes them.
extern "C" int pbx_corpus_append_device(pbx_corpus* c, const int64_t* d_image_ids, const uint8_t* d_hashes, uint64_t n, void* cuda_stream) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (n == 0) return PBX_OK;
    if (!d_image_ids || !d_hashes) return fail(PBX_E_INVALID, "NULL ids or hashes with n > 0");
    std::lock_guard<std::mutex> alk(c->append_mu);
    CU_TRY(cudaSetDevice(c->device));
    int rc = flush_pending_locked(c);
    if (rc != PBX_OK) return rc;
    const uint64_t at = c->n.load();
    if (at + n > c->capacity) {
        if (c->use_vmm) {
            rc = grow_mapped(c, at + n);
        } else {
            std::lock_guard<std::mutex> lk(c->mu);
            rc = reserve_rows(c, at + n);
        }
        if (rc != PBX_OK) return rc;
    }
    cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : c->copy_stream;
    // tight [n][dim] rows -> pitched rows (the padding of fresh capacity is zero already)
    CU_TRY(cudaMemcpy2DAsync(c->d_rows + at * c->pitch, c->pitch, d_hashes, c->dim, c->dim, n, cudaMemcpyDeviceToDevice, s));
    CU_TRY(cudaMemcpyAsync(c->d_ids + at, d_image_ids, n * sizeof(int64_t), cudaMemcpyDeviceToDevice, s));
    row_meta_kernel<<<(unsigned)((n + 7) / 8), 256, 0, s>>>(reinterpret_cast<const uint4*>(c->d_rows), c->pitch16, c->dim, at, n, c->d_inv, c->d_rsum);
    const uint64_t b0 = at / 32, b1 = (at + n + 31) / 32;
    block_meta_kernel<<<(unsigned)((b1 - b0 + 7) / 8), 256, 0, s>>>(c->d_inv, c->d_rsum, c->dim, b0, b1 - b0, at + n, c->d_bmeta);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(s));
    c->n.store(at + n);
    return PBX_OK;
}

extern "C" int pbx_corpus_load(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (n && (!image_ids || !hashes)) return fail(PBX_E_INVALID, "NULL ids or hashes with n > 0");
    std::lock_guard<std::mutex> alk(c->append_mu);  // held across the reset and the upload: no append can land in between
    {
        std::lock_guard<std::mutex> lk(c->mu);
        CU_TRY(cudaSetDevice(c->device));
        CU_TRY(cudaDeviceSynchronize());
        c->n.store(0);
        c->pend_ids.clear(); c->pend_rows.clear(); c->pending.store(0);
    }
    return n ? append_locked(c, image_ids, hashes, n) : PBX_OK;
}

extern "C" int pbx_corpus_fill_synthetic(pbx_corpus* c, uint64_t n, uint64_t seed, uint64_t first_row) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    std::lock_guard<std::mutex> alk(c->append_mu);
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    CU_TRY(cudaDeviceSynchronize());
    c->n.store(0);
    c->pend_ids.clear(); c->pend_rows.clear(); c->pending.store(0);
    int rc = c->use_vmm ? grow_mapped(c, std::max<uint64_t>(n, 1)) : reserve_rows(c, std::max<uint64_t>(n, 1));
    if (rc != PBX_OK) return rc;
    if (n == 0) return PBX_OK;
    const uint64_t step = 1ull << 24;               // rows per launch
    for (uint64_t off = 0; off < n; off += step) {
        const uint64_t m = std::min<uint64_t>(step, n - off);
        synth_fill_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(c->d_rows, c->pitch, c->dim, off, m, seed, first_row + off, c->d_ids);
        const unsigned blocks = (unsigned)((m + 7) / 8);
        row_meta_kernel<<<blocks, 256, 0, c->stream>>>(reinterpret_cast<const uint4*>(c->d_rows), c->pitch16, c->dim, off, m, c->d_inv, c->d_rsum);
        const uint64_t b0 = off / 32, b1 = (off + m + 31) / 32;
        block_meta_kernel<<<(unsigned)((b1 - b0 + 7) / 8), 256, 0, c->stream>>>(c->d_inv, c->d_rsum, c->dim, b0, b1 - b0, off + m, c->d_bmeta);
    }
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaStreamSynchronize(c->stream));
    c->n.store(n);
    return PBX_OK;
}

extern "C" int pbx_corpus_read_rows(const pbx_corpus* cc, uint64_t first, uint64_t n, int64_t* image_ids, uint8_t* hashes) {
    pbx_corpus* c = const_cast<pbx_corpus*>(cc);
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    { int frc = flush_pending(c); if (frc != PBX_OK) return frc; }
    const uint64_t size_now = c->n.load();
    if (n > size_now || first > size_now - n) return fail(PBX_E_INVALID, "rows [%llu, %llu) outside the corpus", (unsigned long long)first, (unsigned long long)(first + n));
    if (n == 0) return PBX_OK;
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    if (image_ids) CU_TRY(cudaMemcpy(image_ids, c->d_ids + first, n * sizeof(int64_t), cudaMemcpyDeviceToHost));
    if (hashes) CU_TRY(cudaMemcpy2D(hashes, c->dim, c->d_rows + first * c->pitch, c->pitch, c->dim, n, cudaMemcpyDeviceToHost));
    return PBX_OK;
}

// ------------------------------------------------------------------------------------------------
// removal
// ------------------------------------------------------------------------------------------------
// The request as the kernels want it: sorted, every id once.  A host std::sort, O(r log r): for large requests it is the
// largest part of the call (tools/remove_time.py).  Ids that are already in order (a folder's ids as SQLite returns them
// from an index, searched again and again) cost one check pass instead.
static int sorted_request(const int64_t* image_ids, uint64_t n, std::vector<int64_t>* out) {
    try { out->assign(image_ids, image_ids + n); } catch (...) { return fail(PBX_E_OOM, "host allocation failed"); }
    if (!std::is_sorted(out->begin(), out->end())) std::sort(out->begin(), out->end());
    out->erase(std::unique(out->begin(), out->end()), out->end());
    return PBX_OK;
}

// Removes every row whose id is in `req` (sorted, unique) by hole filling from the tail (remove.cuh).  Locks as
// pbx_corpus_load does: the pending appends are flushed first, so they are subject to the removal; with mu held no search
// can be enqueued, and the removal stream waits for the last one already enqueued (ev_chain: every search waits for its
// predecessor, so for all of them) before it touches a row.  The new n is published after the stream is synchronised.
static int remove_sorted(pbx_corpus* c, const std::vector<int64_t>& req, uint64_t* out_removed) {
    std::lock_guard<std::mutex> alk(c->append_mu);
    int rc = flush_pending_locked(c);
    if (rc != PBX_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    const uint64_t n = c->n.load();
    if (n == 0 || req.empty()) return PBX_OK;
    cudaStream_t s = c->copy_stream;
    if (c->chain_valid) CU_TRY(cudaStreamWaitEvent(s, c->ev_chain, 0));
    const uint64_t tiles = (n + kRemoveTileRows - 1) / kRemoveTileRows;
    // scratch, stream-ordered (no device-wide synchronisation): [request][removed rows u64, pairs u32][flag words][tile counts x 2]
    const size_t req_bytes = req.size() * sizeof(int64_t), flag_bytes = (n + 31) / 32 * sizeof(uint32_t);
    const size_t off_cnt = (req_bytes + 15) / 16 * 16, off_flags = off_cnt + 16, off_tiles = off_flags + (flag_bytes + 15) / 16 * 16;
    unsigned char* scratch = nullptr;
    uint32_t* pairs = nullptr;
    CU_TRY(cudaMallocAsync(reinterpret_cast<void**>(&scratch), off_tiles + 2 * tiles * sizeof(uint32_t), s));
    int64_t* d_req = reinterpret_cast<int64_t*>(scratch);
    u64* d_removed = reinterpret_cast<u64*>(scratch + off_cnt);
    uint32_t* d_pairs = reinterpret_cast<uint32_t*>(scratch + off_cnt + 8);
    uint32_t* d_flags = reinterpret_cast<uint32_t*>(scratch + off_flags);
    uint32_t* d_tile_holes = reinterpret_cast<uint32_t*>(scratch + off_tiles);
    uint32_t* d_tile_srcs = d_tile_holes + tiles;
    u64 m = 0;
    cudaError_t e = cudaMemcpyAsync(d_req, req.data(), req_bytes, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(d_removed, 0, sizeof(u64), s);
    if (e == cudaSuccess) {
        mark_ids_kernel<<<(unsigned)tiles, kRemoveTileRows, 0, s>>>(c->d_ids, n, d_req, req.size(), 0u, d_flags, d_removed);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&m, d_removed, sizeof(u64), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);        // the one synchronisation before the end: m sizes the rest
    if (e == cudaSuccess && m > n) { cudaFreeAsync(scratch, s); cudaStreamSynchronize(s); return fail(PBX_E_INTERNAL, "removal counted %llu of %llu rows", (unsigned long long)m, (unsigned long long)n); }
    const uint64_t n_keep = n - m;
    // holes below n_keep == survivors at or above it, at most min(m, n_keep): the exact number stays on the device
    const uint64_t max_pairs = std::min<uint64_t>(m, n_keep);
    if (e == cudaSuccess && max_pairs) e = cudaMallocAsync(reinterpret_cast<void**>(&pairs), 2 * max_pairs * sizeof(uint32_t), s);
    if (e == cudaSuccess && max_pairs) {
        uint32_t* d_holes = pairs;
        uint32_t* d_srcs = pairs + max_pairs;
        remove_count_kernel<<<(unsigned)tiles, kRemoveTileRows, 0, s>>>(d_flags, n, n_keep, d_tile_holes, d_tile_srcs);
        remove_scan_kernel<<<1, 1024, 0, s>>>(d_tile_holes, d_tile_srcs, (uint32_t)tiles, d_pairs);
        remove_place_kernel<<<(unsigned)tiles, kRemoveTileRows, 0, s>>>(d_flags, n, n_keep, d_tile_holes, d_tile_srcs, d_holes, d_srcs);
        const uint64_t chunks = max_pairs * c->pitch16;
        const unsigned grid = (unsigned)std::min<uint64_t>((chunks + 255) / 256, (uint64_t)c->sm_count * 8);
        remove_move_kernel<<<grid, 256, 0, s>>>(d_holes, d_srcs, d_pairs, c->pitch16, reinterpret_cast<uint4*>(c->d_rows), c->d_ids, c->d_inv, c->d_rsum);
        e = cudaGetLastError();
    }
    // A moved row may lie outside its new block's {norm, rowterm} range, and the batched epilogue trusts that range as a
    // bound: recompute every block below n_keep (8 bytes per row), the last one over the rows below n_keep only.
    if (e == cudaSuccess && m && n_keep) {
        const uint64_t blocks = (n_keep + 31) / 32;
        block_meta_kernel<<<(unsigned)((blocks + 7) / 8), 256, 0, s>>>(c->d_inv, c->d_rsum, c->dim, 0, blocks, n_keep, c->d_bmeta);
        e = cudaGetLastError();
    }
    if (pairs) cudaFreeAsync(pairs, s);
    cudaFreeAsync(scratch, s);
    const cudaError_t e2 = cudaStreamSynchronize(s);
    if (e == cudaSuccess) e = e2;
    // on failure n stays: the rows below it may be half moved, but a CUDA error here leaves the context unusable anyway
    if (e != cudaSuccess) return fail(PBX_E_CUDA, "removal failed: %s", cudaGetErrorString(e));
    c->n.store(n_keep);
    if (out_removed) *out_removed = m;
    return PBX_OK;
}

extern "C" int pbx_corpus_remove(pbx_corpus* c, const int64_t* image_ids, uint64_t n, uint64_t* out_removed) {
    if (out_removed) *out_removed = 0;
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (n && !image_ids) return fail(PBX_E_INVALID, "NULL image_ids with n > 0");
    if (n == 0) return PBX_OK;
    std::vector<int64_t> req;
    int rc = sorted_request(image_ids, n, &req);
    return rc == PBX_OK ? remove_sorted(c, req, out_removed) : rc;
}

// ------------------------------------------------------------------------------------------------
// replacement
// ------------------------------------------------------------------------------------------------
// The request as the kernels want it: ids sorted, every id once with the hash of its LAST occurrence (what a sequence of
// UPDATE statements leaves), and [ids.size()][pitch] rows in that order with zero padding.  Sorting (id, position) pairs
// puts the last occurrence at the end of each run; ids already strictly in order skip the sort.
struct ReplaceRequest {
    std::vector<int64_t> ids;
    std::vector<uint8_t> rows;
};
static int replace_request(const int64_t* image_ids, const uint8_t* hashes, uint64_t n, uint32_t dim, uint32_t pitch, ReplaceRequest* out) {
    if (n > PBX_MAX_ROWS) return fail(PBX_E_INVALID, "replace request of %llu ids (max %llu)", (unsigned long long)n, (unsigned long long)PBX_MAX_ROWS);
    try {
        std::vector<std::pair<int64_t, uint32_t>> order(n);
        for (uint64_t i = 0; i < n; ++i) order[i] = {image_ids[i], (uint32_t)i};
        if (std::adjacent_find(image_ids, image_ids + n, [](int64_t a, int64_t b) { return a >= b; }) != image_ids + n)
            std::sort(order.begin(), order.end());
        out->ids.clear();
        for (uint64_t i = 0; i < n; ++i)
            if (i + 1 == n || order[i + 1].first != order[i].first) out->ids.push_back(order[i].first);
        out->rows.assign(out->ids.size() * (size_t)pitch, 0);
        for (uint64_t i = 0, j = 0; i < n; ++i)
            if (i + 1 == n || order[i + 1].first != order[i].first) memcpy(out->rows.data() + (j++) * pitch, hashes + (size_t)order[i].second * dim, dim);
    } catch (...) { return fail(PBX_E_OOM, "host allocation failed"); }
    return PBX_OK;
}

// Writes the request's hash into every row whose id it lists, in place (replace.cuh).  Locks and orders as remove_sorted:
// the pending appends are flushed first, so they are subject to the replacement; with mu held no search can be enqueued,
// and the stream waits for the last one already enqueued (ev_chain) before it touches a row.  Returns after the stream is
// synchronised.  Positions, ids and n do not change.
static int replace_sorted(pbx_corpus* c, const ReplaceRequest& req, uint64_t* out_replaced) {
    std::lock_guard<std::mutex> alk(c->append_mu);
    int rc = flush_pending_locked(c);
    if (rc != PBX_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    const uint64_t n = c->n.load(), u = req.ids.size();
    if (n == 0 || u == 0) return PBX_OK;
    cudaStream_t s = c->copy_stream;
    if (c->chain_valid) CU_TRY(cudaStreamWaitEvent(s, c->ev_chain, 0));
    const unsigned tiles = (unsigned)((n + kMarkTileRows - 1) / kMarkTileRows);
    // scratch, stream-ordered: [request ids][request rows][counts: pairs, blocks], then the pair and block lists sized for
    // one row per id (ids are unique in the table the corpus caches); more matches size them exactly and mark once more
    const size_t off_rows = (u * sizeof(int64_t) + 15) / 16 * 16, off_cnt = off_rows + u * c->pitch;
    unsigned char* scratch = nullptr;
    unsigned char* lists = nullptr;
    uint64_t cap = std::min<uint64_t>(n, u);
    uint32_t counts[2] = {0, 0};
    CU_TRY(cudaMallocAsync(reinterpret_cast<void**>(&scratch), off_cnt + 16, s));
    int64_t* d_req = reinterpret_cast<int64_t*>(scratch);
    uint32_t* d_counts = reinterpret_cast<uint32_t*>(scratch + off_cnt);
    cudaError_t e = cudaMemcpyAsync(d_req, req.ids.data(), u * sizeof(int64_t), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(scratch + off_rows, req.rows.data(), u * c->pitch, cudaMemcpyHostToDevice, s);
    for (int pass = 0; pass < 2 && e == cudaSuccess; ++pass) {
        e = cudaMallocAsync(reinterpret_cast<void**>(&lists), cap * (sizeof(uint2) + sizeof(uint32_t)), s);
        if (e == cudaSuccess) e = cudaMemsetAsync(d_counts, 0, 2 * sizeof(uint32_t), s);
        if (e == cudaSuccess) {
            replace_mark_kernel<<<tiles, kMarkTileRows, 0, s>>>(c->d_ids, n, d_req, u, (uint32_t)cap, reinterpret_cast<uint2*>(lists),
                                                                reinterpret_cast<uint32_t*>(lists + cap * sizeof(uint2)), d_counts);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(counts, d_counts, sizeof(counts), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);    // the count sizes the rest (a second time only if ids repeat)
        if (e != cudaSuccess || counts[0] <= cap) break;
        cudaFreeAsync(lists, s);
        lists = nullptr;
        cap = counts[0];
    }
    const uint64_t m = counts[0], blocks = counts[1];
    if (e == cudaSuccess && (m > cap || blocks > m)) {
        if (lists) cudaFreeAsync(lists, s);
        cudaFreeAsync(scratch, s);
        cudaStreamSynchronize(s);
        return fail(PBX_E_INTERNAL, "replacement counted %llu rows in %llu blocks of %llu rows", (unsigned long long)m, (unsigned long long)blocks, (unsigned long long)n);
    }
    if (e == cudaSuccess && m) {
        const uint2* d_pairs = reinterpret_cast<const uint2*>(lists);
        const uint32_t* d_blocks = reinterpret_cast<const uint32_t*>(lists + cap * sizeof(uint2));
        const uint64_t chunks = m * c->pitch16;
        const unsigned grid = (unsigned)std::min<uint64_t>((chunks + 255) / 256, (uint64_t)c->sm_count * 8);
        replace_write_kernel<<<grid, 256, 0, s>>>(d_pairs, m, reinterpret_cast<const uint4*>(scratch + off_rows), c->pitch16, reinterpret_cast<uint4*>(c->d_rows));
        replace_row_meta_kernel<<<(unsigned)((m + 7) / 8), 256, 0, s>>>(d_pairs, m, reinterpret_cast<const uint4*>(c->d_rows), c->pitch16, c->dim, c->d_inv, c->d_rsum);
        replace_block_meta_kernel<<<(unsigned)((blocks + 7) / 8), 256, 0, s>>>(d_blocks, blocks, c->d_inv, c->d_rsum, c->dim, n, c->d_bmeta);
        e = cudaGetLastError();
    }
    if (lists) cudaFreeAsync(lists, s);
    cudaFreeAsync(scratch, s);
    const cudaError_t e2 = cudaStreamSynchronize(s);
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) return fail(PBX_E_CUDA, "replacement failed: %s", cudaGetErrorString(e));
    if (out_replaced) *out_replaced = m;
    return PBX_OK;
}

extern "C" int pbx_corpus_replace(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n, uint64_t* out_replaced) {
    if (out_replaced) *out_replaced = 0;
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (n && (!image_ids || !hashes)) return fail(PBX_E_INVALID, "NULL ids or hashes with n > 0");
    if (n == 0) return PBX_OK;
    ReplaceRequest req;
    int rc = replace_request(image_ids, hashes, n, c->dim, c->pitch, &req);
    return rc == PBX_OK ? replace_sorted(c, req, out_replaced) : rc;
}

// ------------------------------------------------------------------------------------------------
// search
// ------------------------------------------------------------------------------------------------
__global__ void empty_result_kernel(pbx_hit* hits, uint32_t* counts, uint32_t nq, uint32_t k) {
    const uint32_t total = nq * k;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        pbx_hit h; h.image_id = INT64_MAX; h.dist = __int_as_float(0x7f800000); h.dot = 0; h.norm2 = 0; h.flags = 0;
        hits[i] = h;
    }
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nq; i += gridDim.x * blockDim.x) counts[i] = 0;
}

// Launch with programmatic stream serialization: the kernel may begin before its predecessor in the stream has
// finished; it orders itself with pdl_wait() (common.cuh).
template <typename P>
static cudaError_t launch_pdl(void (*kern)(const P), int grid, int block, size_t smem, cudaStream_t s, const P& params) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, params);
}

// RESTRICT: the fast pass of a filtered or paged search (scan_kernel's RESTRICT instantiations); the exact pass and the
// generic kernel test p.allow and p.cut at run time.
template <bool EXACT, bool RESTRICT>
static cudaError_t launch_scan_as(const pbx_corpus* c, const ScanParams& p, int grid, size_t smem, cudaStream_t s) {
    static_assert(!(EXACT && RESTRICT), "the exact pass has no RESTRICT instantiation");
#define PBX_SCAN_CASE(LL, CC)                                                                                                     \
    {                                                                                                                             \
        return launch_pdl<ScanParams>(scan_kernel<LL, CC, EXACT, scan_minb(LL * CC), false, RESTRICT>, grid, kScanThreads, smem, s, p); \
    }
    switch (c->pitch16) {
        case 1: PBX_SCAN_CASE(1, 1)
        case 2: PBX_SCAN_CASE(2, 1)
        case 4: PBX_SCAN_CASE(4, 1)
        case 8: PBX_SCAN_CASE(8, 1)
        case 16:
            if constexpr (!EXACT) {                  // occupancy variants of the d=256 fast pass (pbx_set_scan_ctas_per_sm)
                if (c->ctas_per_sm == 3 || c->ctas_per_sm == 0) return launch_pdl<ScanParams>(scan_kernel<16, 1, false, 3, false, RESTRICT>, grid, kScanThreads, smem, s, p);
                if (c->ctas_per_sm >= 4) return launch_pdl<ScanParams>(scan_kernel<16, 1, false, 4, false, RESTRICT>, grid, kScanThreads, smem, s, p);
            }
            PBX_SCAN_CASE(16, 1)
        case 32: PBX_SCAN_CASE(32, 1)
        case 64: PBX_SCAN_CASE(32, 2)
        case 128: PBX_SCAN_CASE(32, 4)
#define PBX_SCAN_CASE_M(LL, CC, MM) case (LL) * (CC): return launch_pdl<ScanParams>(scan_kernel<LL, CC, EXACT, MM, false, RESTRICT>, grid, kScanThreads, smem, s, p);
        PBX_EXTRA_SHAPES(PBX_SCAN_CASE_M)
#undef PBX_SCAN_CASE_M
        default: {
            if constexpr (!EXACT) {
                // any other row length: the smallest lane layout that holds it, with the row stride at run time
#define PBX_SCAN_CASE_R(LL, CC, MM) \
    if (c->pitch16 <= (LL) * (CC)) return launch_pdl<ScanParams>(scan_kernel<LL, CC, false, MM, true, RESTRICT>, grid, kScanThreads, smem, s, p);
                PBX_RAGGED_SHAPES(PBX_SCAN_CASE_R)
#undef PBX_SCAN_CASE_R
            }
            size_t sm = smem + (size_t)c->pitch16 * 32;               // the exact pass of those shapes: one lane per row
            return launch_pdl<ScanParams>(scan_generic_kernel<EXACT>, grid, kScanThreads, sm, s, p);
        }
    }
#undef PBX_SCAN_CASE
}

template <bool EXACT>
static cudaError_t launch_scan(const pbx_corpus* c, const ScanParams& p, int grid, size_t smem, cudaStream_t s) {
    if constexpr (!EXACT) {
        if (p.allow || p.cut) return launch_scan_as<false, true>(c, p, grid, smem, s);
    }
    return launch_scan_as<EXACT, false>(c, p, grid, smem, s);
}

// true for the row pitches with a compile-time lane layout (1, 3, 5, 6, 8 times a power of two, see scan.cuh)
static bool fast_shape(uint32_t pitch16) {
    if ((pitch16 & (pitch16 - 1)) == 0 && pitch16 <= 256) return true;
#define PBX_IS_SHAPE(LL, CC, MM) if (pitch16 == (LL) * (CC)) return true;
    PBX_EXTRA_SHAPES(PBX_IS_SHAPE)
#undef PBX_IS_SHAPE
    return false;
}

static int scan_grid(const pbx_corpus* c) {
    // 3 CTAs per SM (<= 80 registers) measured best for 256-byte rows; larger rows need the registers, smaller ones fit 4
    const bool pow2 = (c->pitch16 & (c->pitch16 - 1)) == 0;
    uint32_t per_sm = c->ctas_per_sm ? c->ctas_per_sm
                      : c->pitch16 >= 256          ? 1u      // 32 lanes x 8 chunks: one CTA per SM has the registers
                      : (c->pitch16 > 128 && !fast_shape(c->pitch16)) ? 1u      // ragged rows in the 32 x 8 layout
                      : (c->pitch16 < 8 && !pow2)  ? 4u      // ragged rows in the 8 x 1 layout
                      : !pow2                      ? 2u      // the x3 / x5 / x6 shapes and the other ragged layouts
                      : (c->pitch16 == 16 || c->pitch16 == 4) ? 3u : (c->pitch16 > 16) ? 2u : 4u;   // measured: dim 64: 3 -> 6.30 TB/s, 4 -> 5.92
    int g = c->sm_count * (int)per_sm;
    return std::min<int>(g, (int)kMaxScanGrid);
}

// ------------------------------------------------------------------------------------------------
// batched (tensor-core) search
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess) fn = (EncodeTiledFn)p;
    }
    return fn;
}

// [rows][pitch] u8 matrix, boxes of {w bytes, box_rows rows}, w-byte swizzle (the UMMA K-major operand layout)
static int make_u8_map(CUtensorMap* m, void* base, uint64_t rows, uint32_t pitch, uint32_t w, uint32_t box_rows) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return fail(PBX_E_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {(cuuint64_t)pitch, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)pitch};
    cuuint32_t box[2] = {w, box_rows};
    cuuint32_t estr[2] = {1, 1};
    const CUtensorMapSwizzle sw = w == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (w == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(PBX_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return PBX_OK;
}

// Shape of one batched launch (batch.cuh): K-chunk width, CTA grouping, resident queries, ring depth.
struct BatchPlan {
    uint32_t cg;        // CTAs per cluster: 2 = cta_group::2 pairs (default), 1 = single CTAs (PBX_BATCH_CG=1)
    uint32_t tn;        // corpus rows per tile (UMMA N)
    uint32_t w, kc;     // K-chunk bytes, chunks per row
    uint32_t qg;        // resident queries per CTA
    uint32_t groups;    // query groups of cg * qg queries
    uint32_t nq_pad;
    uint32_t stages;
    size_t smem;
    int grid;
};

static bool batch_plan(const pbx_corpus* c, uint32_t nq, uint32_t cg, BatchPlan* out) {
    BatchPlan bp;
    const uint32_t pitch = c->pitch;
    if (pitch % 32 != 0 || pitch > 1024) return false;
    bp.cg = cg;
    bp.tn = 256u;                                    // 256-row tiles: 128 rows per CTA of a pair, all 256 in a single CTA
    bp.w = pitch % 128 == 0 ? 128u : (pitch % 64 == 0 ? 64u : 32u);
    bp.kc = pitch / bp.w;
    const uint32_t stage_bytes = (bp.tn / bp.cg) * bp.w;
    // resident queries per CTA: what the batch needs, at most 512 and at most 128 KB; fewer if the corpus ring would not
    // fit (with more than one 128-query block per CTA a tile must stay resident until the last block has used it)
    uint32_t want = ((nq + bp.cg - 1) / bp.cg + 127u) / 128u * 128u;
    uint32_t qg = std::min<uint32_t>(std::min<uint32_t>(want, kBatchMaxQG), std::max<uint32_t>(128u, (128u * 1024u / pitch) / 128u * 128u));
    for (;; qg -= 128) {
        const size_t fixed = 1024 + (size_t)qg * pitch + batch_smem_fixed(qg, bp.tn);
        if (fixed < kBatchSmemLimit) {
            const uint32_t stages = (uint32_t)std::min<size_t>(kBatchMaxStages, (kBatchSmemLimit - fixed) / stage_bytes);
            const uint32_t need = qg > 128 ? bp.kc + 1 : 2u;
            if (stages >= need) {
                bp.qg = qg; bp.stages = stages; bp.smem = fixed + (size_t)stages * stage_bytes;
                break;
            }
        }
        if (qg == 128) return false;
    }
    bp.groups = (nq + bp.cg * bp.qg - 1) / (bp.cg * bp.qg);
    bp.nq_pad = bp.groups * bp.cg * bp.qg;
    const uint32_t clusters = std::max<uint32_t>(bp.groups, ((uint32_t)c->sm_count / bp.cg) / bp.groups * bp.groups);
    bp.grid = (int)(clusters * bp.cg);
    *out = bp;
    return true;
}

// Candidate buffer entries per query.
static uint32_t batch_cap_for(uint32_t keep) { return keep * 8u <= kBatchCap ? kBatchCap : kBatchCapLarge; }

// The seed pass samples up to kBatchSeedTiles complete tiles, evenly strided over the shard: one bound per (query,
// 32-row block), at least `keep` of them per query or there is no starting threshold.
static void batch_seed_geometry(uint32_t n, uint32_t tn, uint32_t* n_tiles, uint32_t* step) {
    const uint32_t full = n / tn;
    *n_tiles = std::min<uint32_t>(full, kBatchSeedTiles);
    *step = *n_tiles ? full / *n_tiles : 1u;
}

// The launch shape of a batch of nq (<= 1024) queries over n rows with `keep` candidates per query, or false if the
// batched path cannot take it.  CTA pairs hold a whole batch of 1024 queries and stream the corpus once; up to 128
// queries fit one CTA, and single CTAs then run twice as many independent tile pipelines (a small batch is bound by the
// per-tile hand-offs between the TMA, MMA and epilogue roles, not by the tensor pipe).  The other grouping is the fallback
// when the preferred one has no shape or too few sample blocks for the seed pass.
static bool batch_choose(const pbx_corpus* c, uint32_t nq, uint32_t n, uint32_t keep, BatchPlan* out) {
    const uint32_t first = c->batch_cg ? c->batch_cg : (nq <= 128u ? 1u : 2u);
    const uint32_t order[2] = {first, 3u - first};
    for (int i = 0; i < (c->batch_cg ? 1 : 2); ++i) {
        BatchPlan bp;
        if (!batch_plan(c, nq, order[i], &bp)) continue;
        // single CTAs hold whole 256-row K-chunks (32 KB at 128-byte chunks): with fewer than four of them in the ring the
        // stream stalls on every tile -- long rows stay on pairs
        if (!c->batch_cg && i == 0 && order[i] == 1u && bp.stages < 4u) continue;
        uint32_t seed_tiles, seed_step;
        batch_seed_geometry(n, bp.tn, &seed_tiles, &seed_step);
        if (seed_tiles * (bp.tn / 32u) < keep + keep / 2u) continue;
        *out = bp;
        return true;
    }
    return false;
}

static bool batch_eligible(const pbx_corpus* c, uint32_t nq, uint32_t n, uint32_t k) {
    // per-query candidate buffers hold kBatchCap keys and are cut back to keep = k + slack at the end: the scheme
    // needs keep well below the capacity, larger k loops over the single-query scan
    const uint32_t keep = batch_keep(k, c->slack);
    BatchPlan bp;
    return nq >= c->batch_min && keep * 8u <= kBatchCapLarge && n <= kBatchMaxRows && batch_choose(c, std::min<uint32_t>(nq, 1024u), n, keep, &bp);
}

static int ensure_batch_scratch(pbx_corpus* c, uint32_t nq_pad, uint32_t cap) {
    if (nq_pad <= c->batch_pad && cap <= c->batch_cap) return PBX_OK;
    nq_pad = std::max(nq_pad, c->batch_pad);
    cap = std::max(cap, c->batch_cap);
    CU_TRY(cudaDeviceSynchronize());
    cudaFree(c->d_qpad); cudaFree(c->d_colterm); cudaFree(c->d_thr); cudaFree(c->d_bcnt); cudaFree(c->d_boverflow); cudaFree(c->d_bcand);
    cudaFree(c->d_bhist); cudaFree(c->d_binvq); c->d_bhist = nullptr; c->d_binvq = nullptr;
    c->d_qpad = nullptr; c->d_colterm = nullptr; c->d_thr = nullptr; c->d_bcnt = nullptr; c->d_boverflow = nullptr; c->d_bcand = nullptr;
    c->batch_pad = 0; c->map_q_pad = 0; c->batch_cap = 0;
    CU_TRY(cudaMalloc(&c->d_qpad, (size_t)nq_pad * c->pitch));
    CU_TRY(cudaMalloc(&c->d_colterm, (size_t)nq_pad * sizeof(int)));
    CU_TRY(cudaMalloc(&c->d_thr, (size_t)nq_pad * sizeof(float)));
    CU_TRY(cudaMalloc(&c->d_bcnt, (size_t)nq_pad * sizeof(uint32_t)));
    CU_TRY(cudaMalloc(&c->d_boverflow, (size_t)nq_pad * sizeof(uint32_t)));
    CU_TRY(cudaMalloc(&c->d_bcand, (size_t)nq_pad * cap * sizeof(u64)));
    CU_TRY(cudaMalloc(&c->d_bhist, (size_t)nq_pad * kBatchHistBins * sizeof(uint32_t)));
    CU_TRY(cudaMalloc(&c->d_binvq, (size_t)nq_pad * sizeof(float)));
    cudaFree(c->d_seedlb); c->d_seedlb = nullptr;
    CU_TRY(cudaMalloc(&c->d_seedlb, (size_t)kBatchSeedTiles * 8u * nq_pad * sizeof(float)));
    c->batch_pad = nq_pad;
    c->batch_cap = cap;
    return PBX_OK;
}

// Staging layout of the finalize kernel: groups of up to kFinalThreads candidates, `slice16` 16-byte chunks of every
// row of the group per round (row stride slice16 * 16 + 16 bytes).  Returns false if not even one chunk fits.
static bool finalize_stage_layout(size_t avail_bytes, uint32_t keep, uint32_t pitch16, uint32_t* group, uint32_t* slice16, size_t* bytes) {
    uint32_t g = std::min<uint32_t>(keep, (uint32_t)kFinalThreads);
    if (g == 0) g = 1;
    while (g > 32 && avail_bytes / g < 48) g /= 2;
    // the row stride is (slice16 + 1) rounded up to an odd number of 16-byte units: reserve 32 bytes beyond the slice
    if (avail_bytes / g < 48) return false;
    const uint32_t s16 = (uint32_t)std::min<size_t>(pitch16, (avail_bytes / g - 32) / 16);
    *group = g; *slice16 = s16; *bytes = (size_t)g * ((size_t)((s16 + 1) | 1u) * 16);
    return s16 >= 1;
}

// The exact (tie-resolving) pass of one query as a pair of launches: the scan that replays every row with
// kappa >= theta, and the merge of its per-CTA lists.  Launched from the device by the finalize kernels when a
// certificate fails; from the host only to repair a refused device-side launch.
// The f32 bound of the exact pass: the smallest float >= max_dist, so that for every f32 dist, dist < bound exactly
// when (double)dist < max_dist (NaN stays NaN: nothing passes, as in the f64 comparison).
static float dist_bound(double max_dist) {
    float f = (float)max_dist;
    if ((double)f < max_dist) f = std::nextafter(f, std::numeric_limits<float>::infinity());
    return f;
}

struct ExactSetup {
    ScanParams scan;
    FinalizeExactParams fin;
    size_t scan_smem, fin_smem;
    int grid;
};

static ExactSetup exact_setup(const pbx_corpus* c, uint32_t q, uint32_t k, double max_dist, uint32_t n, pbx_hit* d_hits, uint32_t* d_count) {
    ExactSetup x;
    memset(&x, 0, sizeof(x));
    x.grid = scan_grid(c);
    const uint32_t cap_scan_x = next_pow2(k + kTileRows);
    const uint32_t cap_merge_x = next_pow2(k + kMergeChunk);
    ScanParams& sp = x.scan;
    sp.rows = reinterpret_cast<const uint4*>(c->d_rows); sp.inv_norm = c->d_inv; sp.ids = c->d_ids; sp.n = n;
    sp.pitch16 = c->pitch16; sp.dim = c->dim;
    sp.q16 = c->d_q16 + (size_t)q * c->pitch; sp.qbytes = c->d_qbytes + (size_t)q * c->pitch; sp.qh = c->d_qh + q;
    sp.keep = k; sp.cap = cap_scan_x; sp.cand = c->d_cand; sp.cand_cnt = c->d_cand_cnt; sp.tile_counter = c->d_tile_counter;
    sp.hist = c->d_hist; sp.status = c->d_status + q; sp.max_dist = dist_bound(max_dist); sp.allow = c->cur_allow;
    sp.cut = c->cur_cut ? c->cur_cut + q : nullptr;
    FinalizeExactParams& xp = x.fin;
    xp.cand = reinterpret_cast<const KeyX*>(c->d_cand); xp.cand_cnt = c->d_cand_cnt; xp.grid = (uint32_t)x.grid; xp.k = k;
    xp.cap = cap_merge_x; xp.dim = c->dim; xp.pitch = c->pitch; xp.rows = c->d_rows; xp.qbytes = sp.qbytes;
    xp.hits = d_hits + (size_t)q * k; xp.count = d_count + q; xp.status = c->d_status + q; xp.tile_counter = c->d_tile_counter;
    xp.exact_passes = c->d_exact_passes;
    xp.done_flag = c->cur_done_flag; xp.done_seq = c->cur_done_seq;
    x.scan_smem = (size_t)cap_scan_x * sizeof(KeyX);
    x.fin_smem = (size_t)cap_merge_x * sizeof(KeyX);
    return x;
}

static ExactLaunch exact_launch(const ExactSetup& x) {
    ExactLaunch l;
    l.scan = x.scan; l.fin = x.fin; l.grid = (uint32_t)x.grid; l.scan_smem = (uint32_t)x.scan_smem; l.fin_smem = (uint32_t)x.fin_smem; l.pad = 0;
    return l;
}

template <int CG, bool SEED>
static cudaError_t launch_batch_mma(const BatchPlan& bp, const BatchMmaParams& mp, cudaStream_t s) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)bp.grid);
    cfg.blockDim = dim3(kBatchThreads);
    cfg.dynamicSmemBytes = bp.smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, batch_mma_kernel<CG, SEED>, mp);
}

// Enqueues the tensor-core search of nq (<= 1024) device-resident queries.  Caller holds c->mu.
static int enqueue_search_batched(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* d_hits,
                                  uint32_t* d_count, cudaStream_t s, uint32_t n) {
    const uint32_t pitch = c->pitch;
    BatchPlan bp;
    const uint32_t keep = batch_keep(k, c->slack);
    if (!batch_choose(c, nq, n, keep, &bp)) return fail(PBX_E_INTERNAL, "batched path: no launch shape for pitch %u", pitch);
    int rc = ensure_query_scratch(c, nq);
    if (rc != PBX_OK) return rc;
    const uint32_t cap = batch_cap_for(keep);
    rc = ensure_batch_scratch(c, bp.nq_pad, cap);
    if (rc != PBX_OK) return rc;
    const uint32_t box_rows = bp.tn / bp.cg, qbox = (bp.qg % 256u) ? 128u : 256u;
    if (c->map_rows_gen != c->rows_generation || c->map_rows_box != box_rows) {
        // with reserved address ranges the map covers the whole range once: tiles beyond the committed rows are never touched
        // (TMA coordinates are signed 32-bit: a row dimension beyond 2^31 makes the copy an illegal instruction)
        rc = make_u8_map(&c->map_rows, c->d_rows, std::min<uint64_t>(c->use_vmm ? c->reserved_rows : c->capacity.load(), kBatchMaxRows), pitch, bp.w, box_rows);
        if (rc != PBX_OK) return rc;
        c->map_rows_gen = c->rows_generation; c->map_rows_box = box_rows;
    }
    if (c->map_q_pad != c->batch_pad || c->map_q_box != qbox) {
        rc = make_u8_map(&c->map_q, c->d_qpad, c->batch_pad, pitch, bp.w, qbox);
        if (rc != PBX_OK) return rc;
        c->map_q_pad = c->batch_pad; c->map_q_box = qbox;
    }
    const int grid_scan = scan_grid(c);
    rc = ensure_cand(c, (size_t)std::max<uint32_t>(keep, k) * grid_scan * sizeof(KeyX));      // exact-pass scratch
    if (rc != PBX_OK) return rc;

    BatchPrepParams pp;
    pp.queries = d_queries; pp.nq = nq; pp.dim = c->dim; pp.pitch = pitch;
    pp.qpad = c->d_qpad; pp.q16 = c->d_q16; pp.qbytes = c->d_qbytes; pp.qh = c->d_qh;
    pp.colterm = c->d_colterm; pp.thr = c->d_thr; pp.cand_cnt = c->d_bcnt; pp.overflow = c->d_boverflow;
    pp.bhist = c->d_bhist; pp.inv_q = c->d_binvq;
    batch_prep_kernel<<<bp.nq_pad, 128, (size_t)c->dim * sizeof(float), s>>>(pp);
    CU_TRY(cudaGetLastError());

    BatchMmaParams mp;
    mp.map_rows = c->map_rows; mp.map_q = c->map_q;
    mp.inv_norm = c->d_inv; mp.row_sum = c->d_rsum; mp.blk_meta = c->d_bmeta; mp.colterm = c->d_colterm; mp.thr = c->d_thr;
    mp.cand = c->d_bcand; mp.cand_cnt = c->d_bcnt; mp.overflow = c->d_boverflow;
    mp.bhist = c->d_bhist; mp.inv_q = c->d_binvq; mp.thr_live = c->d_thr; mp.keep = keep; mp.cap = cap;
    mp.n = n; mp.dim = c->dim; mp.w = bp.w; mp.kc = bp.kc; mp.qg = bp.qg; mp.groups = bp.groups; mp.stages = bp.stages; mp.tn = bp.tn;
    mp.seed_lb = c->d_seedlb; mp.nq_pad = bp.nq_pad; mp.allow = c->cur_allow; mp.cut = c->cur_cut;
    // L2 prefetch ahead of the shared-memory ring: measured counter-productive (10M x 256, 8 queries: 0.55 ms without, 0.56 /
    // 0.73 / 0.78 ms at 6 / 12 / 24 tiles ahead) -- the small-batch pass is bound by the MMA thread's serial
    // wait -> issue -> commit loop per 128-row tile, not by the stream.  Kept as an experiment knob, off.
    mp.prefetch_tiles = getenv("PBX_BATCH_PREFETCH") ? (uint32_t)atoi(getenv("PBX_BATCH_PREFETCH")) : 0u;
    mp.exp_flags = getenv("PBX_BATCH_EXPFLAGS") ? (uint32_t)atoi(getenv("PBX_BATCH_EXPFLAGS")) : 0u;
    BatchTightenParams tp;
    tp.cand = c->d_bcand; tp.cand_cnt = c->d_bcnt; tp.thr = c->d_thr; tp.keep = keep; tp.nq = nq; tp.cap = cap;

    // 1. seed pass over a strided sample of complete tiles: one bound per (query, 32-row block), nothing is pushed
    uint32_t seed_tiles, seed_step;
    batch_seed_geometry(n, bp.tn, &seed_tiles, &seed_step);
    mp.n_tiles = seed_tiles; mp.tile_step = seed_step; mp.tile_base = 0;
    CU_TRY((bp.cg == 2 ? launch_batch_mma<2, true>(bp, mp, s) : launch_batch_mma<1, true>(bp, mp, s)));
    // 2. starting threshold of every query = its keep-th largest bound
    BatchSeedSelectParams sp;
    sp.seed_lb = c->d_seedlb; sp.n_blocks = seed_tiles * (bp.tn / 32u); sp.nq_pad = bp.nq_pad; sp.keep = keep; sp.thr = c->d_thr;
    batch_seed_select_kernel<<<nq, 256, (size_t)sp.n_blocks * sizeof(u64), s>>>(sp);
    CU_TRY(cudaGetLastError());
    if (getenv("PBX_BATCH_EXP")) {
        // experiment: the bare pipeline (TMA, MMA, TMEM loads, max trees; nothing stored) over every tile
        BatchMmaParams xp = mp;
        xp.seed_lb = nullptr; xp.n_tiles = (n + bp.tn - 1) / bp.tn; xp.tile_step = 1; xp.tile_base = 0;
        CU_TRY((bp.cg == 2 ? launch_batch_mma<2, true>(bp, xp, s) : launch_batch_mma<1, true>(bp, xp, s)));
    }
    // 3. the main pass over every tile; thresholds keep tightening from the per-query histograms of accepted keys.
    // 4. cut every buffer back to keep: the finalize kernels take at most `keep` candidates per query.
    // A query accepts about keep * (1 + ln(rows / sample rows)) keys over a pass (more while a threshold lags): with the large
    // candidate sets of k ~ 1000 that outgrows the 16384-entry buffers somewhere near 100M rows, and an overflowed buffer
    // costs its query an exact pass over the whole shard (100M x 256, k = 1000: 7.5 s per 1024 queries instead of 75 ms).
    // So long shards run the pass in segments with the cut-back in between: the buffers start every segment at `keep`
    // entries, the thresholds carry over.
    const uint32_t all_tiles = (n + bp.tn - 1) / bp.tn;
    // Segment lengths for keep > 512, from what a buffer can take: a segment may add room = (cap - keep) / (1.5 keep) times
    // keep keys per query (1.5: thresholds lag behind the rows).  The first segment starts from the seed thresholds (the
    // keep-th best of the sample): keep * (1 + ln(rows / sample rows)) keys; a later one from exact thresholds over the rows
    // so far: keep * ln(rows after / rows before).  keep = 1250: the 25M-row cap decides; keep = 2000: 2.9M rows first.
    const double room = (double)(cap - std::min(cap, keep)) / (1.5 * (double)keep);
    const double first_tiles = (double)std::max<uint32_t>(seed_tiles, 1u) * std::exp(std::max(0.0, std::min(room - 1.0, 20.0)));
    const double growth = std::exp(std::min(room, 20.0)) - 1.0;
    uint32_t forced_seg = 0;
    if (const char* e = getenv("PBX_BATCH_SEG_TILES")) forced_seg = std::max<uint32_t>(1u, (uint32_t)atoll(e));    // tests: segments on small shards
    mp.tile_step = 1;
    for (uint32_t t0 = 0; t0 < all_tiles;) {
        uint32_t seg = all_tiles - t0;
        if (forced_seg) seg = std::min(seg, forced_seg);
        else if (keep > 512u) {
            const double lim = t0 == 0 ? first_tiles : (double)t0 * growth;
            seg = std::min<uint32_t>(seg, (uint32_t)std::max(256.0, std::min(lim, (double)kBatchSegTilesLarge)));
        }
        mp.tile_base = t0; mp.n_tiles = seg;
        CU_TRY((bp.cg == 2 ? launch_batch_mma<2, false>(bp, mp, s) : launch_batch_mma<1, false>(bp, mp, s)));
        batch_tighten_kernel<<<nq, 256, (size_t)cap * sizeof(u64), s>>>(tp);
        CU_TRY(cudaGetLastError());
        t0 += seg;
    }

    // per-query finalize: bit-exact re-rank, certificate; exact passes are tail-launched by its last CTA
    const ExactSetup xs = exact_setup(c, 0, k, max_dist, n, d_hits, d_count);       // template of query 0
    if (keep <= kBfThreads) {
        BatchFinalizeParams fp;
        memset(&fp, 0, sizeof(fp));
        fp.x = exact_launch(xs);
        fp.bcand = c->d_bcand; fp.bcnt = c->d_bcnt; fp.boverflow = c->d_boverflow; fp.bticket = c->d_tile_counter + 100;
        fp.bcap = cap; fp.nq = nq; fp.keep = keep; fp.k = k; fp.n = n; fp.n_allowed = c->cur_allowed; fp.cut = c->cur_cut; fp.dim = c->dim; fp.pitch = pitch;
        fp.rows = c->d_rows; fp.ids = c->d_ids; fp.qbytes = c->d_qbytes; fp.q16 = c->d_q16; fp.qh = c->d_qh;
        fp.max_dist = max_dist; fp.margin = certificate_margin(c->dim);
        fp.hits = d_hits; fp.count = d_count; fp.status = c->d_status;
        batch_finalize_kernel<<<nq, (keep + 31u) & ~31u, batch_finalize_smem(pitch), s>>>(fp);
        CU_TRY(cudaGetLastError());
    } else {
        const uint32_t chunk = kFinalThreads;
        const uint32_t cap_merge = std::max<uint32_t>(next_pow2(keep + chunk), kBatchCap);     // >= candidates left per query
        const size_t off_sorted = (size_t)cap_merge * sizeof(u64);
        const size_t off_dots = 2 * off_sorted;
        const size_t off_q = (off_dots + (size_t)keep * 20 + 15) & ~(size_t)15;
        const size_t off_stage = (off_q + (size_t)pitch * 6 + 15) & ~(size_t)15;
        const size_t fin_budget = 200 * 1024;
        uint32_t stage_rows = 0, slice16 = 0;
        size_t stage_bytes = 0;
        if (off_stage >= fin_budget || !finalize_stage_layout(fin_budget - off_stage, keep, pitch / 16, &stage_rows, &slice16, &stage_bytes))
            return fail(PBX_E_INTERNAL, "finalize layout does not fit shared memory (k=%u dim=%u)", k, c->dim);
        const size_t fin_smem = off_stage + stage_bytes;
        FinalizeParams fp;
        memset(&fp, 0, sizeof(fp));
        fp.grid = (uint32_t)grid_scan; fp.keep = keep; fp.cap = cap_merge; fp.chunk = chunk; fp.k = k; fp.n = n; fp.n_allowed = c->cur_allowed; fp.cut = c->cur_cut;
        fp.dim = c->dim; fp.pitch = pitch; fp.stage_rows = stage_rows; fp.slice16 = slice16;
        fp.off_sorted = (uint32_t)off_sorted; fp.off_ent = 0; fp.off_dots = (uint32_t)off_dots; fp.off_q = (uint32_t)off_q; fp.off_stage = (uint32_t)off_stage;
        fp.rows = c->d_rows; fp.ids = c->d_ids; fp.qbytes = c->d_qbytes; fp.q16 = c->d_q16; fp.qh = c->d_qh;
        fp.max_dist = max_dist; fp.margin = certificate_margin(c->dim);
        fp.hits = d_hits; fp.count = d_count; fp.status = c->d_status; fp.tile_counter = c->d_tile_counter;
        fp.hist = c->d_hist; fp.cand = nullptr; fp.cand_cnt = nullptr;
        fp.bcand = c->d_bcand; fp.bcnt = c->d_bcnt; fp.boverflow = c->d_boverflow; fp.bticket = c->d_tile_counter + 100;
        fp.bcap = cap; fp.nq = nq;
        fp.x = exact_launch(xs);
        finalize_kernel<true><<<nq, kFinalThreads, fin_smem, s>>>(fp);
        CU_TRY(cudaGetLastError());
    }
#ifndef PBX_USE_CDP
    // build without device-side launches (sanitizer runs): the host reads the certificates and launches the exact passes
    {
        std::vector<SearchStatus> hs(nq);
        CU_TRY(cudaStreamSynchronize(s));
        CU_TRY(cudaMemcpy(hs.data(), c->d_status, (size_t)nq * sizeof(SearchStatus), cudaMemcpyDeviceToHost));
        for (uint32_t q = 0; q < nq; ++q) {
            if (!hs[q].need_exact) continue;
            const ExactSetup xq = exact_setup(c, q, k, max_dist, n, d_hits, d_count);
            CU_TRY(launch_scan<true>(c, xq.scan, xq.grid, xq.scan_smem, s));
            finalize_exact_kernel<<<1, kFinalThreads, xq.fin_smem, s>>>(xq.fin);
            CU_TRY(cudaGetLastError());
        }
    }
#endif
    c->batched_queries += nq;
    c->last_grid = bp.grid;
    return PBX_OK;
}

// A search restricted to a set of image ids (pbx_search_filtered and its twins).
struct SearchFilter {
    const int64_t* ids;     // ascending, duplicates allowed: host memory, or device memory if `device`
    uint64_t n;
    uint32_t mode;          // PBX_FILTER_INCLUDE / PBX_FILTER_EXCLUDE
    bool device;            // device ids: their order is checked on the device (PBX_COUNT_FILTER_UNSORTED)
};

static int check_filter_args(const int64_t* ids, uint64_t n, uint32_t mode) {
    if (n && !ids) return fail(PBX_E_INVALID, "filter_ids is NULL with n_filter = %llu", (unsigned long long)n);
    if (mode != PBX_FILTER_INCLUDE && mode != PBX_FILTER_EXCLUDE) return fail(PBX_E_INVALID, "unknown filter mode %u", mode);
    if (n > PBX_MAX_ROWS) return fail(PBX_E_INVALID, "n_filter = %llu exceeds PBX_MAX_ROWS", (unsigned long long)n);
    return PBX_OK;
}

// The filter of a host-form call: the ids sorted and deduplicated into *sorted.  *out = NULL for an empty EXCLUDE set,
// which is an unfiltered search.
static int host_filter(const int64_t* ids, uint64_t n, uint32_t mode, std::vector<int64_t>* sorted, SearchFilter* f, const SearchFilter** out) {
    *out = nullptr;
    int rc = check_filter_args(ids, n, mode);
    if (rc != PBX_OK) return rc;
    if (mode == PBX_FILTER_EXCLUDE && n == 0) return PBX_OK;
    if (n) { rc = sorted_request(ids, n, sorted); if (rc != PBX_OK) return rc; }
    f->ids = sorted->data(); f->n = sorted->size(); f->mode = mode; f->device = false;
    *out = f;
    return PBX_OK;
}

// Stream-ordered mark pass of a filtered search over rows [0, n): the row bitmap and the allowed count, both corpus
// scratch that the next search on any stream only touches after this one (ev_chain).  Caller holds c->mu.
static int enqueue_filter_mark(pbx_corpus* c, const SearchFilter& f, uint32_t n, cudaStream_t s) {
    const size_t words = ((size_t)n + kTileRows - 1) / kTileRows * kTileRows / 32;    // every row a kernel may look at
    int rc = ensure_filter_scratch(c, std::max<size_t>(words, 1), f.device ? 0 : f.n);
    if (rc != PBX_OK) return rc;
    const int64_t* d_set = f.ids;
    if (!f.device && f.n) {
        CU_TRY(cudaMemcpyAsync(c->d_filter_ids, f.ids, f.n * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        d_set = c->d_filter_ids;
    }
    CU_TRY(cudaMemsetAsync(c->d_filter_words, 0, 2 * sizeof(u64), s));
    if (f.device && f.n > 1) {
        const unsigned blocks = (unsigned)std::min<uint64_t>((f.n + 255) / 256, (uint64_t)c->sm_count * 8);
        ids_unsorted_kernel<<<blocks, 256, 0, s>>>(d_set, f.n, reinterpret_cast<uint32_t*>(c->d_filter_words + 1));
        CU_TRY(cudaGetLastError());
    }
    if (n) {
        mark_ids_kernel<<<(n + kMarkTileRows - 1) / kMarkTileRows, kMarkTileRows, 0, s>>>(c->d_ids, n, d_set, f.n,
                                                                                       f.mode == PBX_FILTER_EXCLUDE ? 1u : 0u, c->d_allow, c->d_filter_words);
        CU_TRY(cudaGetLastError());
    }
    c->cur_allow = c->d_allow;
    c->cur_allowed = c->d_filter_words;
    return PBX_OK;
}

// Enqueues the whole search for nq queries already on the device.  Caller holds c->mu.
static int enqueue_search(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* d_hits,
                          uint32_t* d_count, cudaStream_t s, bool timed, uint32_t* done_flag = nullptr, uint32_t done_seq = 0,
                          const SearchFilter* filter = nullptr, const pbx_hit* after = nullptr, bool after_on_device = false) {
    const uint32_t n = (uint32_t)c->n.load();
    c->cur_done_flag = done_flag; c->cur_done_seq = done_seq;    // only the single-query kernels publish to it
    c->cur_allow = nullptr; c->cur_allowed = nullptr; c->cur_cut = nullptr;
    c->last_n = n;
    c->scan_timed = false;
    if (c->chain_valid) CU_TRY(cudaStreamWaitEvent(s, c->ev_chain, 0));
    if (timed) CU_TRY(cudaEventRecord(c->ev_t0, s));
    if (filter) {
        int rc = enqueue_filter_mark(c, *filter, n, s);
        if (rc != PBX_OK) return rc;
    }
    PageCut* cuts = nullptr;                                    // paged search: one cut per query, derived on the device
    if (after) {
        int rc = ensure_page_scratch(c, nq);
        if (rc != PBX_OK) return rc;
        cuts = c->d_cut;
        const pbx_hit* d_after = after;
        if (!after_on_device) {                                 // host cursors: a stream-ordered copy into corpus scratch
            CU_TRY(cudaMemcpyAsync(c->d_after, after, (size_t)nq * sizeof(pbx_hit), cudaMemcpyHostToDevice, s));
            d_after = c->d_after;
        }
        page_cut_kernel<<<(nq + 255) / 256, 256, 0, s>>>(d_after, nq, (double)certificate_margin(c->dim), c->d_cut);
        CU_TRY(cudaGetLastError());
    }
    if (n == 0) {
        empty_result_kernel<<<64, 256, 0, s>>>(d_hits, d_count, nq, k);
        CU_TRY(cudaGetLastError());
    } else if (batch_eligible(c, nq, n, k)) {
        for (uint32_t q0 = 0; q0 < nq; q0 += 1024) {
            const uint32_t b = std::min<uint32_t>(1024u, nq - q0);
            c->cur_cut = cuts ? cuts + q0 : nullptr;
            int rc = enqueue_search_batched(c, d_queries + (size_t)q0 * c->dim, b, k, max_dist, d_hits + (size_t)q0 * k, d_count + q0, s, n);
            if (rc != PBX_OK) return rc;
        }
    } else {
        int rc = ensure_query_scratch(c, nq);
        if (rc != PBX_OK) return rc;
        const int grid = scan_grid(c);
        const uint32_t keep = std::min<uint32_t>(default_keep(k, c->slack), kMaxKeep);
        // fast pass: room for two rounds of pushes, so the flood before the first global threshold needs no cut-back
        const uint32_t cap_scan = next_pow2(keep + 2 * kTileRows);
        const int seed_grid = c->sm_count;
        const bool seeded = (uint64_t)n >= (uint64_t)seed_grid * kSeedThreads * 8;       // small shards: not worth a launch
        // merge round size: one element per thread, more only when a round must span a complete rank (2 * grid)
        const uint32_t chunk = std::min<uint32_t>(4u, std::max<uint32_t>(1u, (2u * (uint32_t)grid + kFinalThreads - 1) / kFinalThreads)) * kFinalThreads;
        const uint32_t cap_merge = next_pow2(keep + chunk);
        rc = ensure_cand(c, (size_t)std::max<uint32_t>(keep, k) * grid * sizeof(KeyX));
        if (rc != PBX_OK) return rc;
        const float margin = certificate_margin(c->dim);
        // finalize kernel shared memory: [buf cap][sorted cap] (re-used for the (dist, id) sort) | per-candidate
        // arrays | decoded + centred query | staged candidate rows
        const size_t off_sorted = (size_t)cap_merge * sizeof(u64);
        const size_t off_dots = 2 * off_sorted;
        const size_t off_q = (off_dots + (size_t)keep * 20 + 15) & ~(size_t)15;
        const size_t off_stage = (off_q + (size_t)c->pitch * 6 + 15) & ~(size_t)15;
        const size_t fin_budget = 200 * 1024;
        uint32_t stage_rows = 0, slice16 = 0;
        size_t stage_bytes = 0;
        if (off_stage >= fin_budget || !finalize_stage_layout(fin_budget - off_stage, keep, c->pitch16, &stage_rows, &slice16, &stage_bytes))
            return fail(PBX_E_INTERNAL, "finalize layout does not fit shared memory (k=%u dim=%u)", k, c->dim);
        const size_t fin_smem = off_stage + stage_bytes;
        c->cur_cut = cuts;                                       // exact_setup offsets it by the query

        for (uint32_t q = 0; q < nq; ++q) {
            ScanParams sp;
            sp.rows = reinterpret_cast<const uint4*>(c->d_rows);
            sp.inv_norm = c->d_inv;
            sp.ids = c->d_ids;
            sp.n = n;
            sp.pitch16 = c->pitch16;
            sp.dim = c->dim;
            sp.q16 = c->d_q16 + (size_t)q * c->pitch;
            sp.qbytes = c->d_qbytes + (size_t)q * c->pitch;
            sp.qh = c->d_qh + q;
            sp.keep = keep;
            sp.cap = cap_scan;
            sp.cand = c->d_cand;
            sp.cand_cnt = c->d_cand_cnt;
            sp.tile_counter = c->d_tile_counter;
            sp.hist = c->d_hist;
            sp.status = c->d_status + q;
            sp.max_dist = dist_bound(max_dist);
            sp.allow = c->cur_allow;
            sp.cut = cuts ? cuts + q : nullptr;
            {
                PrepSeedParams ps;
                ps.query = d_queries + (size_t)q * c->dim;
                ps.dim = c->dim; ps.pitch = c->pitch; ps.pitch16 = c->pitch16;
                ps.q16 = c->d_q16 + (size_t)q * c->pitch;
                ps.qbytes = c->d_qbytes + (size_t)q * c->pitch;
                ps.qh = c->d_qh + q;
                ps.rows = sp.rows; ps.inv_norm = sp.inv_norm; ps.n = n; ps.keep = keep;
                ps.do_seed = seeded ? 1u : 0u;
                ps.seed_hist = c->d_hist + kHistBins; ps.ticket = c->d_tile_counter + 96; ps.gbin = c->d_tile_counter + 32;
                ps.allow = c->cur_allow;
                ps.cut = sp.cut;
                CU_TRY(launch_pdl<PrepSeedParams>(prep_seed_kernel, seeded ? seed_grid : 1, kSeedThreads, (size_t)c->pitch * 2, s, ps));
            }
            const bool time_scan = timed && q + 1 == nq;
            if (time_scan) CU_TRY(cudaEventRecord(c->ev_s0, s));
            CU_TRY(launch_scan<false>(c, sp, grid, (size_t)cap_scan * sizeof(u64), s));
            if (time_scan) { CU_TRY(cudaEventRecord(c->ev_s1, s)); c->scan_timed = true; }

            FinalizeParams fp;
            fp.cand = reinterpret_cast<const u64*>(c->d_cand);
            fp.cand_cnt = c->d_cand_cnt;
            fp.grid = (uint32_t)grid;
            fp.keep = keep;
            fp.cap = cap_merge;
            fp.k = k;
            fp.n = n;
            fp.n_allowed = c->cur_allowed;
            fp.cut = sp.cut;
            fp.dim = c->dim;
            fp.pitch = c->pitch;
            fp.rows = c->d_rows;
            fp.ids = c->d_ids;
            fp.qbytes = sp.qbytes;
            fp.q16 = sp.q16;
            fp.chunk = chunk;
            fp.hist = c->d_hist;
            fp.stage_rows = stage_rows;
            fp.slice16 = slice16;
            fp.off_sorted = (uint32_t)off_sorted;
            fp.off_ent = 0;
            fp.off_dots = (uint32_t)off_dots;
            fp.off_q = (uint32_t)off_q;
            fp.off_stage = (uint32_t)off_stage;
            fp.qh = c->d_qh + q;
            fp.max_dist = max_dist;
            fp.margin = margin;
            fp.hits = d_hits + (size_t)q * k;
            fp.count = d_count + q;
            fp.status = c->d_status + q;
            fp.tile_counter = c->d_tile_counter;
            fp.done_flag = c->cur_done_flag; fp.done_seq = c->cur_done_seq;
            // exact pass parameters: k entries per CTA, (dist, image_id) keys
            const ExactSetup xs = exact_setup(c, q, k, max_dist, n, d_hits, d_count);
            const ScanParams& spx = xs.scan;
            const FinalizeExactParams& xp = xs.fin;
            (void)spx; (void)xp;
            fp.x = exact_launch(xs);
            // Long rows or many candidates: one SM would replay keep * dim elements alone (instruction bound, ~0.15 us
            // per candidate-KB).  Split: candidate selection -> replay on keep / 32 CTAs -> order, filter, certificate.
            fp.phase = 0;
            fp.x_keys = reinterpret_cast<u64*>(c->d_split);
            fp.x_sbs = reinterpret_cast<float*>(c->d_split + (size_t)kMaxKeep * 8);
            fp.x_fdots = fp.x_sbs + kMaxKeep;
            fp.x_dots = reinterpret_cast<int*>(fp.x_fdots + kMaxKeep);
            fp.x_norms = fp.x_dots + kMaxKeep;
            fp.x_meta = reinterpret_cast<uint32_t*>(fp.x_norms + kMaxKeep);
            if (c->split_finalize && (size_t)keep * c->pitch >= c->split_min_bytes) {
                fp.phase = 1;
                CU_TRY(launch_pdl<FinalizeParams>(finalize_kernel<false>, 1, kFinalThreads, fin_smem, s, fp));
                ReplayParams rp;
                rp.keys = fp.x_keys; rp.meta = fp.x_meta; rp.rows = c->d_rows; rp.qbytes = sp.qbytes; rp.q16 = sp.q16; rp.qh = sp.qh;
                rp.dim = c->dim; rp.pitch = c->pitch;
                rp.sbs = fp.x_sbs; rp.fdots = fp.x_fdots; rp.dots = fp.x_dots; rp.norms = fp.x_norms;
                const size_t rsm = (size_t)c->pitch * 6 + (size_t)kReplayRows * (kReplaySlice16 + 2) * 16;
                replay_kernel<<<(keep + kReplayRows - 1) / kReplayRows, kReplayThreads, rsm, s>>>(rp);
                CU_TRY(cudaGetLastError());
                fp.phase = 2;
                finalize_kernel<false><<<1, kFinalThreads, fin_smem, s>>>(fp);
                CU_TRY(cudaGetLastError());
            } else {
                CU_TRY(launch_pdl<FinalizeParams>(finalize_kernel<false>, 1, kFinalThreads, fin_smem, s, fp));
            }
#ifndef PBX_USE_CDP
            // without device-side launch both kernels are enqueued always and return at once unless need_exact was raised
            CU_TRY(launch_scan<true>(c, spx, grid, xs.scan_smem, s));
            finalize_exact_kernel<<<1, kFinalThreads, xs.fin_smem, s>>>(xp);
            CU_TRY(cudaGetLastError());
#endif
        }
        c->last_grid = grid;
    }
    if (filter && filter->device) {
        // after every kernel of the search, tail-launched exact passes included: an unsorted filter voids every count
        filter_unsorted_count_kernel<<<(nq + 255) / 256, 256, 0, s>>>(reinterpret_cast<const uint32_t*>(c->d_filter_words + 1), d_count, nq,
                                                                      PBX_COUNT_FILTER_UNSORTED);
        CU_TRY(cudaGetLastError());
    }
    if (timed) CU_TRY(cudaEventRecord(c->ev_t1, s));
    CU_TRY(cudaEventRecord(c->ev_chain, s));
    c->chain_valid = true;
    c->queries += nq;
    c->last_bytes = (uint64_t)n * c->dim * nq;
    return PBX_OK;
}

static int check_search_args(const pbx_corpus* c, const void* queries, uint32_t nq, uint32_t k) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (nq && !queries) return fail(PBX_E_INVALID, "queries is NULL");
    if (k == 0) return fail(PBX_E_INVALID, "k must be >= 1");
    if (k > PBX_MAX_K) return fail(PBX_E_K, "k = %u exceeds PBX_MAX_K = %u", k, PBX_MAX_K);
    return PBX_OK;
}

// after: the cursors of a paged search (NULL: first pages), in device memory if after_on_device, else in host memory.
static int search_device_impl(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* d_hits,
                              uint32_t* d_count, void* cuda_stream, const SearchFilter* filter, const pbx_hit* after = nullptr,
                              bool after_on_device = false) {
    int rc = check_search_args(c, d_queries, nq, k);
    if (rc != PBX_OK) return rc;
    if (nq == 0) return PBX_OK;
    if (!d_hits || !d_count) return fail(PBX_E_INVALID, "NULL output");
    rc = flush_pending(c);                          // coalesced appends become visible before the search (append lock only)
    if (rc != PBX_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : c->stream;
    return enqueue_search(c, d_queries, nq, k, max_dist, d_hits, d_count, s, false, nullptr, 0, filter, after, after_on_device);
}

extern "C" int pbx_search_device(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* d_hits,
                                 uint32_t* d_count, void* cuda_stream) {
    return search_device_impl(c, d_queries, nq, k, max_dist, d_hits, d_count, cuda_stream, nullptr);
}

extern "C" int pbx_search_device_filtered(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* d_hits,
                                          uint32_t* d_count, void* cuda_stream, const int64_t* d_filter_ids, uint64_t n_filter,
                                          uint32_t filter_mode) {
    int rc = check_filter_args(d_filter_ids, n_filter, filter_mode);
    if (rc != PBX_OK) return rc;
    const SearchFilter f = {d_filter_ids, n_filter, filter_mode, true};
    // an empty EXCLUDE set is the unfiltered search
    return search_device_impl(c, d_queries, nq, k, max_dist, d_hits, d_count, cuda_stream,
                              filter_mode == PBX_FILTER_EXCLUDE && n_filter == 0 ? nullptr : &f);
}

static int search_hits_impl(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* out_hits,
                            uint32_t* out_count, const SearchFilter* filter, const pbx_hit* after = nullptr) {
    int rc = check_search_args(c, queries, nq, k);
    if (rc != PBX_OK) return rc;
    if (nq == 0) return PBX_OK;
    if (!out_hits || !out_count) return fail(PBX_E_INVALID, "NULL output");
    rc = flush_pending(c);                          // coalesced appends become visible before the search (append lock only)
    if (rc != PBX_OK) return rc;
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    const uint32_t batch_max = 1024;
    float total_ms = 0.f;
    uint64_t total_bytes = 0;
    for (uint32_t q0 = 0; q0 < nq; q0 += batch_max) {
        const uint32_t b = std::min<uint32_t>(batch_max, nq - q0);
        rc = ensure_query_scratch(c, b);
        if (rc != PBX_OK) return rc;
        rc = ensure_hits(c, (size_t)b * k, b);
        if (rc != PBX_OK) return rc;
        const size_t qbytes = (size_t)b * c->dim;
        if (qbytes > c->h_queries_cap) {
            cudaFreeHost(c->h_queries); c->h_queries = nullptr; c->h_queries_cap = 0;
            CU_TRY(cudaMallocHost(&c->h_queries, std::max<size_t>(qbytes, 64 * 1024)));
            c->h_queries_cap = std::max<size_t>(qbytes, 64 * 1024);
        }
        memcpy(c->h_queries, queries + (size_t)q0 * c->dim, qbytes);
        // One query on the scan path: the kernels write the k records and the count straight into pinned memory and then
        // publish a sequence number this thread polls: no copy-engine operation and no stream synchronisation between the
        // last kernel and the caller (measured: 6-15 us of a 0.44 ms call).  The query still goes through a staged copy:
        // letting the 148 CTAs of the first kernel read it from host memory cost 16 us MORE, and carrying it in the launch
        // parameters made no measurable difference.
        const uint32_t n_now0 = (uint32_t)c->n.load();
        const bool direct = c->zero_copy && b == 1 && n_now0 > 0 && !batch_eligible(c, 1, n_now0, k);
        const uint8_t* q_dev = c->d_queries;
        pbx_hit* hits_dev = c->d_hits;
        if (direct) {
            void* dh = nullptr;
            if (cudaHostGetDevicePointer(&dh, c->h_hits, 0) == cudaSuccess) hits_dev = static_cast<pbx_hit*>(dh);
            else cudaGetLastError();
        }
        const bool polled = direct && hits_dev != c->d_hits;
        CU_TRY(cudaMemcpyAsync(c->d_queries, c->h_queries, qbytes, cudaMemcpyHostToDevice, c->stream));
        // hits and counts share one buffer ([b*k] records, then [b] counts): one copy back
        uint32_t* d_cnt = reinterpret_cast<uint32_t*>(hits_dev + (size_t)b * k);
        uint32_t* h_cnt = reinterpret_cast<uint32_t*>(c->h_hits + (size_t)b * k);
        const size_t back_bytes = (size_t)b * k * sizeof(pbx_hit) + (size_t)b * sizeof(uint32_t);
        uint32_t* flag_dev = nullptr;
        if (polled) {
            void* df = nullptr;
            if (cudaHostGetDevicePointer(&df, c->h_flag, 0) != cudaSuccess) return fail(PBX_E_CUDA, "completion flag is not device-visible");
            flag_dev = static_cast<uint32_t*>(df);
            ++c->flag_seq;
        }
        rc = enqueue_search(c, q_dev, b, k, max_dist, hits_dev, d_cnt, c->stream, c->profiling, flag_dev, c->flag_seq, filter,
                            after ? after + q0 : nullptr);
        if (rc != PBX_OK) return rc;
        if (polled) {
            // spin on the sequence number; look at the stream now and then so that a faulted kernel cannot hang the caller
            volatile uint32_t* flag = c->h_flag;
            for (uint32_t spins = 1; *flag != c->flag_seq; ++spins) {
                if ((spins & 0xFFFFu) == 0) {
                    const cudaError_t qe = cudaStreamQuery(c->stream);
                    if (qe == cudaSuccess) break;                       // everything ran: the word is there (or the answer is incomplete)
                    if (qe != cudaErrorNotReady) return fail(PBX_E_CUDA, "search failed: %s", cudaGetErrorString(qe));
                }
            }
            std::atomic_thread_fence(std::memory_order_acquire);
            if (*flag != c->flag_seq) return fail(PBX_E_INTERNAL, "search finished without publishing its result");
            if (c->profiling) CU_TRY(cudaEventSynchronize(c->ev_t1));
        } else {
            CU_TRY(cudaMemcpyAsync(c->h_hits, c->d_hits, back_bytes, cudaMemcpyDeviceToHost, c->stream));
            CU_TRY(cudaStreamSynchronize(c->stream));
        }
        // A refused device-side launch of the exact pass leaves the uncertified fast-pass hits and a marker in the count:
        // run that query's exact pass from the host (its status still says need_exact, theta is in place) and fetch again.
        {
            uint32_t failed = 0;
            const uint32_t n_now = (uint32_t)c->n.load();
            for (uint32_t q = 0; q < b; ++q) {
                if (h_cnt[q] != PBX_COUNT_EXACT_LAUNCH_FAILED) continue;
                c->cur_done_flag = nullptr;
                const ExactSetup xs = exact_setup(c, q, k, max_dist, std::min<uint32_t>(n_now, c->last_n), hits_dev, d_cnt);
                CU_TRY(launch_scan<true>(c, xs.scan, xs.grid, xs.scan_smem, c->stream));
                finalize_exact_kernel<<<1, kFinalThreads, xs.fin_smem, c->stream>>>(xs.fin);
                CU_TRY(cudaGetLastError());
                ++failed;
            }
            if (failed) {
                if (!polled) CU_TRY(cudaMemcpyAsync(c->h_hits, c->d_hits, back_bytes, cudaMemcpyDeviceToHost, c->stream));
                CU_TRY(cudaStreamSynchronize(c->stream));
                for (uint32_t q = 0; q < b; ++q)
                    if (h_cnt[q] > k) return fail(PBX_E_INTERNAL, "exact pass of query %u could not be completed", q0 + q);
            }
        }
        if (c->profiling) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, c->ev_t0, c->ev_t1) == cudaSuccess) total_ms += ms;
            if (!c->scan_timed || cudaEventElapsedTime(&c->last_scan_ms, c->ev_s0, c->ev_s1) != cudaSuccess) { c->last_scan_ms = 0.f; cudaGetLastError(); }
        }
        total_bytes += c->last_bytes;
        memcpy(out_hits + (size_t)q0 * k, c->h_hits, (size_t)b * k * sizeof(pbx_hit));
        memcpy(out_count + q0, h_cnt, (size_t)b * sizeof(uint32_t));
    }
    c->last_search_ms = total_ms;
    c->last_bytes = total_bytes;
    return PBX_OK;
}

extern "C" int pbx_search_hits(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, pbx_hit* out_hits,
                               uint32_t* out_count) {
    return search_hits_impl(c, queries, nq, k, max_dist, out_hits, out_count, nullptr);
}

// [nq][k] records -> the column outputs of pbx_search (slots past a query's count are zero)
static void split_hits(const std::vector<pbx_hit>& hits, uint32_t k, const uint32_t* out_count, int64_t* out_ids, float* out_dist,
                       int32_t* out_dot, int32_t* out_norm2) {
    for (size_t i = 0; i < hits.size(); ++i) {
        const bool valid = (i % k) < out_count[i / k];
        out_ids[i] = valid ? hits[i].image_id : 0;
        if (out_dist) out_dist[i] = valid ? hits[i].dist : 0.f;
        if (out_dot) out_dot[i] = valid ? hits[i].dot : 0;
        if (out_norm2) out_norm2[i] = valid ? hits[i].norm2 : 0;
    }
}

static int search_impl(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, int64_t* out_ids,
                       float* out_dist, int32_t* out_dot, int32_t* out_norm2, uint32_t* out_count, const SearchFilter* filter) {
    int rc = check_search_args(c, queries, nq, k);
    if (rc != PBX_OK) return rc;
    if (nq == 0) return PBX_OK;
    if (!out_ids || !out_count) return fail(PBX_E_INVALID, "NULL output");
    std::vector<pbx_hit> hits;
    try { hits.resize((size_t)nq * k); } catch (...) { return fail(PBX_E_OOM, "host allocation failed"); }
    rc = search_hits_impl(c, queries, nq, k, max_dist, hits.data(), out_count, filter);
    if (rc != PBX_OK) return rc;
    split_hits(hits, k, out_count, out_ids, out_dist, out_dot, out_norm2);
    return PBX_OK;
}

extern "C" int pbx_search(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, int64_t* out_ids,
                          float* out_dist, int32_t* out_dot, int32_t* out_norm2, uint32_t* out_count) {
    return search_impl(c, queries, nq, k, max_dist, out_ids, out_dist, out_dot, out_norm2, out_count, nullptr);
}

extern "C" int pbx_search_filtered(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, int64_t* out_ids,
                                   float* out_dist, int32_t* out_dot, int32_t* out_norm2, uint32_t* out_count,
                                   const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode) {
    std::vector<int64_t> sorted;
    SearchFilter f;
    const SearchFilter* fp = nullptr;
    int rc = host_filter(filter_ids, n_filter, filter_mode, &sorted, &f, &fp);
    if (rc != PBX_OK) return rc;
    return search_impl(c, queries, nq, k, max_dist, out_ids, out_dist, out_dot, out_norm2, out_count, fp);
}

// ---- paged searches ------------------------------------------------------------------------------------------------------
// A NaN dist is no position in the (dist, image_id) order: the host forms reject it (the device form gives count 0).
static int check_page_args(const pbx_hit* after, uint32_t nq) {
    if (!after) return PBX_OK;
    for (uint32_t i = 0; i < nq; ++i)
        if (std::isnan(after[i].dist)) return fail(PBX_E_INVALID, "after[%u].dist is NaN", i);
    return PBX_OK;
}

// The filter and cursor checks shared by the host forms of a paged search.
static int host_page(const pbx_hit* after, uint32_t nq, const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode,
                     std::vector<int64_t>* sorted, SearchFilter* f, const SearchFilter** fp) {
    int rc = host_filter(filter_ids, n_filter, filter_mode, sorted, f, fp);
    if (rc != PBX_OK) return rc;
    return check_page_args(after, nq);
}

extern "C" int pbx_search_page(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, const pbx_hit* after,
                               const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode, pbx_hit* out_hits, uint32_t* out_count) {
    std::vector<int64_t> sorted;
    SearchFilter f;
    const SearchFilter* fp = nullptr;
    int rc = host_page(after, nq, filter_ids, n_filter, filter_mode, &sorted, &f, &fp);
    if (rc != PBX_OK) return rc;
    return search_hits_impl(c, queries, nq, k, max_dist, out_hits, out_count, fp, after);
}

extern "C" int pbx_search_device_page(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist,
                                      const pbx_hit* d_after, const int64_t* d_filter_ids, uint64_t n_filter, uint32_t filter_mode,
                                      pbx_hit* d_hits, uint32_t* d_count, void* cuda_stream) {
    int rc = check_filter_args(d_filter_ids, n_filter, filter_mode);
    if (rc != PBX_OK) return rc;
    const SearchFilter f = {d_filter_ids, n_filter, filter_mode, true};
    return search_device_impl(c, d_queries, nq, k, max_dist, d_hits, d_count, cuda_stream,
                              filter_mode == PBX_FILTER_EXCLUDE && n_filter == 0 ? nullptr : &f, d_after, true);
}

extern "C" int pbx_merge_hits(const pbx_hit* gathered, const uint32_t* counts, uint32_t n_shards, uint32_t nq, uint32_t k,
                              pbx_hit* out_hits, uint32_t* out_count) {
    if (!gathered || !counts || !out_hits || !out_count) return fail(PBX_E_INVALID, "NULL argument");
    if (k == 0 || n_shards == 0) return fail(PBX_E_INVALID, "k and n_shards must be >= 1");
    std::vector<uint32_t> head;
    try { head.resize(n_shards); } catch (...) { return fail(PBX_E_OOM, "host allocation failed"); }
    for (uint32_t q = 0; q < nq; ++q) {
        std::fill(head.begin(), head.end(), 0u);
        uint32_t out = 0;
        while (out < k) {
            int best = -1;
            const pbx_hit* bh = nullptr;
            for (uint32_t s = 0; s < n_shards; ++s) {
                const uint32_t cnt = std::min<uint32_t>(counts[(size_t)s * nq + q], k);
                if (head[s] >= cnt) continue;
                const pbx_hit* h = gathered + ((size_t)s * nq + q) * k + head[s];
                // (dist as f64, image_id) ascending: the ORDER BY of src/engine.rs:380 with ties by id
                if (!bh || (double)h->dist < (double)bh->dist || ((double)h->dist == (double)bh->dist && h->image_id < bh->image_id)) {
                    bh = h;
                    best = (int)s;
                }
            }
            if (best < 0) break;
            out_hits[(size_t)q * k + out++] = *bh;
            head[best]++;
        }
        out_count[q] = out;
        for (uint32_t i = out; i < k; ++i) {
            pbx_hit h; h.image_id = INT64_MAX; h.dist = std::numeric_limits<float>::infinity(); h.dot = 0; h.norm2 = 0; h.flags = 0;
            out_hits[(size_t)q * k + i] = h;
        }
    }
    return PBX_OK;
}

extern "C" int pbx_merge_hits_device(int device, const pbx_hit* d_gathered, const uint32_t* d_counts, uint32_t n_shards, uint32_t nq,
                                     uint32_t k, pbx_hit* d_out_hits, uint32_t* d_out_count, void* cuda_stream) {
    if (!d_gathered || !d_out_hits || !d_out_count) return fail(PBX_E_INVALID, "NULL argument");
    if (k == 0 || n_shards == 0 || n_shards > PBX_MAX_SHARDS) return fail(PBX_E_INVALID, "k >= 1 and 1 <= n_shards <= %u required", PBX_MAX_SHARDS);
    if (nq == 0) return PBX_OK;
    CU_TRY(cudaSetDevice(device));
    const uint32_t stage = merge_smem_bytes(n_shards, k);
    static std::atomic<uint64_t> attr_done{0};                   // one bit per device: the attribute is per device context
    if (device >= 0 && device < 64 && !((attr_done.load(std::memory_order_acquire) >> device) & 1ull)) {
        CU_TRY(cudaFuncSetAttribute(merge_hits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMergeSmemKeys * 12u)));
        attr_done.fetch_or(1ull << device, std::memory_order_release);
    } else if (device < 0 || device >= 64) {
        CU_TRY(cudaFuncSetAttribute(merge_hits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMergeSmemKeys * 12u)));
    }
    merge_hits_kernel<<<nq, kMergeThreads, stage, static_cast<cudaStream_t>(cuda_stream)>>>(d_gathered, d_counts, n_shards, nq, k, d_out_hits,
                                                                                           d_out_count, stage);
    CU_TRY(cudaGetLastError());
    return PBX_OK;
}

// ------------------------------------------------------------------------------------------------
// peer-memory exchange (multi-GPU merge step)
// ------------------------------------------------------------------------------------------------
struct pbx_exchange {
    int device = 0;
    uint32_t rank = 0, world = 1;
    uint32_t max_records = 0, max_queries = 0;
    uint32_t slot_records = 0, slot_flags = 0;
    size_t mail_bytes = 0, bytes = 0;
    void* base = nullptr;                          // [2 slots][world][max_records] records, then [2][max_queries][world] flags
    void* peer_base[PBX_MAX_SHARDS] = {};
    bool connected = false;
    uint32_t seq = 0;
    pbx_hit* d_out = nullptr;                      // merged result of pbx_exchange_search_hits: [max_records] records, then [max_queries] counts
    pbx_hit* h_out = nullptr;                      // pinned
    size_t out_records = 0;
    uint32_t* h_flag = nullptr;                    // pinned: [0] completion sequence number, [1] the shard's own count (zero-copy completion)
    uint32_t flag_seq = 0;
    // set around the launch by pbx_exchange_search_hits for a one-query call (see ExchangeParams)
    const uint32_t* zc_local_count = nullptr;
    uint32_t* zc_local_count_out = nullptr;
    uint32_t* zc_flag = nullptr;
};

extern "C" int pbx_exchange_create(int device, uint32_t rank, uint32_t world, uint32_t max_records, uint32_t max_queries, pbx_exchange** out) {
    if (!out) return fail(PBX_E_INVALID, "out is NULL");
    *out = nullptr;
    if (world == 0 || world > PBX_MAX_SHARDS || rank >= world || max_records == 0 || max_queries == 0)
        return fail(PBX_E_INVALID, "bad exchange geometry (rank %u of %u)", rank, world);
    if (pbx_device_count() == 0) return fail(PBX_E_NO_DEVICE, "no sm_100 device: pixelbox_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaFuncSetAttribute(exchange_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(kMergeSmemKeys * 12u)));
    pbx_exchange* x = new (std::nothrow) pbx_exchange();
    if (!x) return fail(PBX_E_OOM, "host allocation failed");
    x->device = device; x->rank = rank; x->world = world; x->max_records = max_records; x->max_queries = max_queries;
    x->slot_records = world * max_records;
    x->slot_flags = max_queries * world;
    x->mail_bytes = ((size_t)2 * x->slot_records * sizeof(pbx_hit) + 255) & ~(size_t)255;
    x->bytes = x->mail_bytes + (size_t)2 * x->slot_flags * sizeof(uint32_t);
    cudaError_t e = cudaMalloc(&x->base, x->bytes);
    if (e == cudaSuccess) e = cudaMemset(x->base, 0, x->bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(x->base);
        cudaGetLastError();
        delete x;
        return fail(e == cudaErrorMemoryAllocation ? PBX_E_OOM : PBX_E_CUDA, "exchange allocation failed: %s", cudaGetErrorString(e));
    }
    *out = x;
    return PBX_OK;
}

extern "C" int pbx_exchange_handle(pbx_exchange* x, void* out_handle) {
    if (!x || !out_handle) return fail(PBX_E_INVALID, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CU_TRY(cudaSetDevice(x->device));
    cudaIpcMemHandle_t h;
    CU_TRY(cudaIpcGetMemHandle(&h, x->base));
    memcpy(out_handle, &h, sizeof(h));
    return PBX_OK;
}

extern "C" int pbx_exchange_connect(pbx_exchange* x, const void* all_handles) {
    if (!x || !all_handles) return fail(PBX_E_INVALID, "NULL argument");
    if (x->connected) return PBX_OK;
    CU_TRY(cudaSetDevice(x->device));
    for (uint32_t r = 0; r < x->world; ++r) {
        if (r == x->rank) { x->peer_base[r] = x->base; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, static_cast<const char*>(all_handles) + (size_t)r * sizeof(h), sizeof(h));
        void* ptr = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return fail(PBX_E_CUDA, "cannot map the mailbox of rank %u (peer access over NVLink required): %s", r, cudaGetErrorString(e));
        x->peer_base[r] = ptr;
    }
    x->connected = true;
    return PBX_OK;
}

extern "C" int pbx_exchange_allgather_merge(pbx_exchange* x, const pbx_hit* d_local, uint32_t nq, uint32_t k, pbx_hit* d_out,
                                            uint32_t* d_out_count, void* cuda_stream) {
    if (!x || !d_local || !d_out || !d_out_count) return fail(PBX_E_INVALID, "NULL argument");
    if (!x->connected) return fail(PBX_E_INVALID, "exchange is not connected");
    if (nq == 0) return PBX_OK;
    if (k == 0 || (uint64_t)nq * k > x->max_records || nq > x->max_queries)
        return fail(PBX_E_INVALID, "exchange sized for %u records / %u queries per call, got %u x %u", x->max_records, x->max_queries, nq, k);
    CU_TRY(cudaSetDevice(x->device));
    ExchangeParams p;
    memset(&p, 0, sizeof(p));
    for (uint32_t r = 0; r < x->world; ++r) {
        p.peer_mail[r] = static_cast<pbx_hit*>(x->peer_base[r]);
        p.peer_flag[r] = reinterpret_cast<uint32_t*>(static_cast<char*>(x->peer_base[r]) + x->mail_bytes);
    }
    p.local = d_local; p.out = d_out; p.out_count = d_out_count;
    p.rank = x->rank; p.world = x->world; p.nq = nq; p.k = k;
    p.seq = x->seq + 1; p.slot = p.seq & 1u;
    p.slot_records = x->slot_records; p.slot_flags = x->slot_flags;
    p.stage_bytes = merge_smem_bytes(x->world, k);
    if (x->zc_flag && nq == 1) { p.local_count = x->zc_local_count; p.local_count_out = x->zc_local_count_out; p.done_flag = x->zc_flag; p.done_seq = x->flag_seq; }
    exchange_merge_kernel<<<nq, kMergeThreads, p.stage_bytes, static_cast<cudaStream_t>(cuda_stream)>>>(p);
    CU_TRY(cudaGetLastError());
    x->seq = p.seq;                                 // only a launched call consumes a sequence number (the ranks stay in step)
    return PBX_OK;
}

// Host buffers in, host buffers out, for one rank of the row-sharded path: H2D of the queries, the shard's local search,
// the fused exchange + merge kernel, D2H of the merged result, one synchronisation -- all on the corpus' stream, no
// other host work in between (the Python driver's torch copies cost ~30 us per query more).  Every rank makes the same
// call with the same queries; every rank receives the global result.
static int exchange_search_hits_impl(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                     pbx_hit* out_hits, uint32_t* out_count, const SearchFilter* filter, const pbx_hit* after = nullptr) {
    if (!x) return fail(PBX_E_INVALID, "exchange is NULL");
    int rc = check_search_args(c, queries, nq, k);
    if (rc != PBX_OK) return rc;
    if (nq == 0) return PBX_OK;
    if (!out_hits || !out_count) return fail(PBX_E_INVALID, "NULL output");
    if (!x->connected) return fail(PBX_E_INVALID, "exchange is not connected");
    if (x->device != c->device) return fail(PBX_E_INVALID, "exchange and corpus live on different devices");
    rc = flush_pending(c);
    if (rc != PBX_OK) return rc;
    if ((uint64_t)nq * k > x->max_records || nq > x->max_queries || nq > 1024)
        return fail(PBX_E_INVALID, "exchange sized for %u records / %u queries per call, got %u x %u", x->max_records, x->max_queries, nq, k);
    std::lock_guard<std::mutex> lk(c->mu);
    CU_TRY(cudaSetDevice(c->device));
    if (!x->d_out) {
        x->out_records = (size_t)x->max_records + ((size_t)x->max_queries * sizeof(uint32_t) + sizeof(pbx_hit) - 1) / sizeof(pbx_hit) + 1;
        CU_TRY(cudaMalloc(&x->d_out, x->out_records * sizeof(pbx_hit)));
        CU_TRY(cudaMallocHost(&x->h_out, x->out_records * sizeof(pbx_hit)));
    }
    rc = ensure_query_scratch(c, nq);
    if (rc != PBX_OK) return rc;
    rc = ensure_hits(c, (size_t)nq * k, nq);
    if (rc != PBX_OK) return rc;
    const size_t qbytes = (size_t)nq * c->dim;
    if (qbytes > c->h_queries_cap) {
        cudaFreeHost(c->h_queries); c->h_queries = nullptr; c->h_queries_cap = 0;
        CU_TRY(cudaMallocHost(&c->h_queries, std::max<size_t>(qbytes, 64 * 1024)));
        c->h_queries_cap = std::max<size_t>(qbytes, 64 * 1024);
    }
    memcpy(c->h_queries, queries, qbytes);
    CU_TRY(cudaMemcpyAsync(c->d_queries, c->h_queries, qbytes, cudaMemcpyHostToDevice, c->stream));
    uint32_t* d_cnt_local = reinterpret_cast<uint32_t*>(c->d_hits + (size_t)nq * k);
    rc = enqueue_search(c, c->d_queries, nq, k, max_dist, c->d_hits, d_cnt_local, c->stream, false, nullptr, 0, filter, after);
    if (rc != PBX_OK) return rc;
    // one query: the merge kernel writes the merged records, both counts and a sequence number into pinned memory and this
    // thread polls it (as pbx_search_hits does on one device); otherwise two copies back and a synchronisation
    pbx_hit* out_dev = x->d_out;
    uint32_t* flag_dev = nullptr;
    uint32_t* local_out_dev = nullptr;
    if (c->zero_copy && nq == 1) {
        if (!x->h_flag) { CU_TRY(cudaMallocHost(&x->h_flag, 64)); x->h_flag[0] = 0; }
        void *dh = nullptr, *df = nullptr;
        if (cudaHostGetDevicePointer(&dh, x->h_out, 0) == cudaSuccess && cudaHostGetDevicePointer(&df, x->h_flag, 0) == cudaSuccess) {
            out_dev = static_cast<pbx_hit*>(dh);
            flag_dev = static_cast<uint32_t*>(df);
            local_out_dev = flag_dev + 1;
        } else {
            cudaGetLastError();
        }
    }
    uint32_t* d_cnt_out = reinterpret_cast<uint32_t*>(out_dev + (size_t)nq * k);
    if (flag_dev) { ++x->flag_seq; x->zc_flag = flag_dev; x->zc_local_count = d_cnt_local; x->zc_local_count_out = local_out_dev; }
    rc = pbx_exchange_allgather_merge(x, c->d_hits, nq, k, out_dev, d_cnt_out, c->stream);
    x->zc_flag = nullptr;
    if (rc != PBX_OK) return rc;
    const size_t out_bytes = (size_t)nq * k * sizeof(pbx_hit) + (size_t)nq * sizeof(uint32_t);
    if (flag_dev) {
        volatile uint32_t* flag = x->h_flag;
        for (uint32_t spins = 1; *flag != x->flag_seq; ++spins) {
            if ((spins & 0xFFFFu) == 0) {
                const cudaError_t qe = cudaStreamQuery(c->stream);
                if (qe == cudaSuccess) break;
                if (qe != cudaErrorNotReady) return fail(PBX_E_CUDA, "sharded search failed: %s", cudaGetErrorString(qe));
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        if (*flag != x->flag_seq) return fail(PBX_E_INTERNAL, "sharded search finished without publishing its result");
        reinterpret_cast<uint32_t*>(c->h_hits)[0] = x->h_flag[1];
    } else {
        CU_TRY(cudaMemcpyAsync(x->h_out, x->d_out, out_bytes, cudaMemcpyDeviceToHost, c->stream));
        // the local counts too: a refused device-side exact launch shows there (PBX_COUNT_EXACT_LAUNCH_FAILED)
        CU_TRY(cudaMemcpyAsync(c->h_hits, d_cnt_local, (size_t)nq * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaStreamSynchronize(c->stream));
    }
    const uint32_t* h_cnt = reinterpret_cast<const uint32_t*>(x->h_out + (size_t)nq * k);
    const uint32_t* h_local = reinterpret_cast<const uint32_t*>(c->h_hits);
    for (uint32_t q = 0; q < nq; ++q) {
        if (h_cnt[q] == PBX_COUNT_EXCHANGE_TIMEOUT) return fail(PBX_E_INTERNAL, "peer exchange timed out: a rank did not post its records");
        if (h_local[q] > k) return fail(PBX_E_INTERNAL, "this shard could not certify query %u (count marker 0x%x)", q, h_local[q]);
    }
    memcpy(out_hits, x->h_out, (size_t)nq * k * sizeof(pbx_hit));
    memcpy(out_count, h_cnt, (size_t)nq * sizeof(uint32_t));
    return PBX_OK;
}

extern "C" int pbx_exchange_search_hits(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                        pbx_hit* out_hits, uint32_t* out_count) {
    return exchange_search_hits_impl(x, c, queries, nq, k, max_dist, out_hits, out_count, nullptr);
}

extern "C" int pbx_exchange_search_hits_filtered(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k,
                                                 double max_dist, pbx_hit* out_hits, uint32_t* out_count, const int64_t* filter_ids,
                                                 uint64_t n_filter, uint32_t filter_mode) {
    std::vector<int64_t> sorted;
    SearchFilter f;
    const SearchFilter* fp = nullptr;
    int rc = host_filter(filter_ids, n_filter, filter_mode, &sorted, &f, &fp);
    if (rc != PBX_OK) return rc;
    return exchange_search_hits_impl(x, c, queries, nq, k, max_dist, out_hits, out_count, fp);
}

extern "C" int pbx_exchange_search_hits_page(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k,
                                             double max_dist, const pbx_hit* after, const int64_t* filter_ids, uint64_t n_filter,
                                             uint32_t filter_mode, pbx_hit* out_hits, uint32_t* out_count) {
    std::vector<int64_t> sorted;
    SearchFilter f;
    const SearchFilter* fp = nullptr;
    int rc = host_page(after, nq, filter_ids, n_filter, filter_mode, &sorted, &f, &fp);
    if (rc != PBX_OK) return rc;
    return exchange_search_hits_impl(x, c, queries, nq, k, max_dist, out_hits, out_count, fp, after);
}

extern "C" void pbx_exchange_destroy(pbx_exchange* x) {
    if (!x) return;
    cudaSetDevice(x->device);
    cudaDeviceSynchronize();
    cudaFree(x->d_out); cudaFreeHost(x->h_out); cudaFreeHost(x->h_flag);
    for (uint32_t r = 0; r < x->world; ++r)
        if (r != x->rank && x->peer_base[r]) cudaIpcCloseMemHandle(x->peer_base[r]);
    cudaFree(x->base);
    cudaGetLastError();
    delete x;
}

extern "C" int pbx_cosine_distance_pairs(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim, float* out_dist,
                                         int32_t* out_dot, int32_t* out_norm2_a, int32_t* out_norm2_b) {
    if (dim == 0 || dim > PBX_MAX_DIM) return fail(PBX_E_DIM, "dim %u outside [1, %u]", dim, PBX_MAX_DIM);
    if (n == 0) return PBX_OK;
    if (!a || !b || !out_dist) return fail(PBX_E_INVALID, "NULL argument");
    if (pbx_device_count() == 0) return fail(PBX_E_NO_DEVICE, "no sm_100 device: pixelbox_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    uint8_t *da = nullptr, *db = nullptr;
    float* dd = nullptr;
    int* di = nullptr;
    int rc = PBX_OK;
    cudaError_t e = cudaMalloc(&da, n * dim);
    if (e == cudaSuccess) e = cudaMalloc(&db, n * dim);
    if (e == cudaSuccess) e = cudaMalloc(&dd, n * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&di, 3 * n * sizeof(int));
    if (e == cudaSuccess) e = cudaMemcpy(da, a, n * dim, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b, n * dim, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        pair_distance_kernel<<<(unsigned)((n + 127) / 128), 128>>>(da, db, n, dim, dd, di, di + n, di + 2 * n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out_dist, dd, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_dot) e = cudaMemcpy(out_dot, di, n * sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_norm2_a) e = cudaMemcpy(out_norm2_a, di + n, n * sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_norm2_b) e = cudaMemcpy(out_norm2_b, di + 2 * n, n * sizeof(int), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = fail(e == cudaErrorMemoryAllocation ? PBX_E_OOM : PBX_E_CUDA, "pair distance failed: %s", cudaGetErrorString(e));
    cudaFree(da); cudaFree(db); cudaFree(dd); cudaFree(di);
    return rc;
}

// byte_distance / hamming_distance for pairs: which = 0 byte, 1 hamming
static int pair_byte_hamming(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim, int which, float* out_dist,
                             uint32_t* out_int) {
    if (dim == 0 || dim > PBX_MAX_DIM) return fail(PBX_E_DIM, "dim %u outside [1, %u]", dim, PBX_MAX_DIM);
    if (n == 0) return PBX_OK;
    if (!a || !b || !out_dist) return fail(PBX_E_INVALID, "NULL argument");
    if (pbx_device_count() == 0) return fail(PBX_E_NO_DEVICE, "no sm_100 device: pixelbox_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    uint8_t *da = nullptr, *db = nullptr;
    float* dd = nullptr;
    uint32_t* di = nullptr;
    cudaError_t e = cudaMalloc(&da, n * dim);
    if (e == cudaSuccess) e = cudaMalloc(&db, n * dim);
    if (e == cudaSuccess) e = cudaMalloc(&dd, n * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&di, n * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMemcpy(da, a, n * dim, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(db, b, n * dim, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        const unsigned blocks = (unsigned)((n * 32 + 255) / 256);
        if (which == 0) pair_byte_hamming_kernel<<<blocks, 256>>>(da, db, n, dim, dd, di, nullptr, nullptr);
        else pair_byte_hamming_kernel<<<blocks, 256>>>(da, db, n, dim, nullptr, nullptr, dd, di);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out_dist, dd, n * sizeof(float), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && out_int) e = cudaMemcpy(out_int, di, n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
    cudaFree(da); cudaFree(db); cudaFree(dd); cudaFree(di);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? PBX_E_OOM : PBX_E_CUDA, "pair distance failed: %s", cudaGetErrorString(e));
    return PBX_OK;
}

extern "C" int pbx_byte_distance_pairs(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim, float* out_dist,
                                       uint32_t* out_l1) {
    if (n > (1ull << 26)) return fail(PBX_E_INVALID, "at most 2^26 pairs per call");
    return pair_byte_hamming(device, a, b, n, dim, 0, out_dist, out_l1);
}

extern "C" int pbx_hamming_distance_pairs(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim, float* out_dist,
                                          uint32_t* out_bits) {
    if (n > (1ull << 26)) return fail(PBX_E_INVALID, "at most 2^26 pairs per call");
    return pair_byte_hamming(device, a, b, n, dim, 1, out_dist, out_bits);
}

extern "C" int pbx_quantize(int device, const float* embeddings, uint64_t n, uint8_t* out) {
    if (n == 0) return PBX_OK;
    if (!embeddings || !out) return fail(PBX_E_INVALID, "NULL argument");
    if (pbx_device_count() == 0) return fail(PBX_E_NO_DEVICE, "no sm_100 device: pixelbox_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    float* din = nullptr;
    uint8_t* dout = nullptr;
    cudaError_t e = cudaMalloc(&din, n * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&dout, n);
    if (e == cudaSuccess) e = cudaMemcpy(din, embeddings, n * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        quantize_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 65535), 256>>>(din, n, dout);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, dout, n, cudaMemcpyDeviceToHost);
    cudaFree(din); cudaFree(dout);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? PBX_E_OOM : PBX_E_CUDA, "quantize failed: %s", cudaGetErrorString(e));
    return PBX_OK;
}

extern "C" int pbx_quantize_device(int device, const float* d_embeddings, uint64_t n, uint8_t* d_out, void* cuda_stream) {
    if (n == 0) return PBX_OK;
    if (!d_embeddings || !d_out) return fail(PBX_E_INVALID, "NULL argument");
    if (pbx_device_count() == 0) return fail(PBX_E_NO_DEVICE, "no sm_100 device: pixelbox_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    quantize_kernel<<<(unsigned)std::min<uint64_t>((n + 255) / 256, 65535), 256, 0, static_cast<cudaStream_t>(cuda_stream)>>>(d_embeddings, n, d_out);
    CU_TRY(cudaGetLastError());
    return PBX_OK;
}

extern "C" int pbx_int8_peak(int device, double* out_tops) {
    if (!out_tops) return fail(PBX_E_INVALID, "out_tops is NULL");
    if (pbx_device_count() == 0) return fail(PBX_E_NO_DEVICE, "no sm_100 device: pixelbox_b200 has no CPU fallback");
    CU_TRY(cudaSetDevice(device));
    int sms = 0;
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    sms &= ~1;
    const size_t smem = 4 * 128 * 128 + 1024;
    CU_TRY(cudaFuncSetAttribute(batch_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)sms);
    cfg.blockDim = dim3(128);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    const int iters = 20000;                         // ~10 ms per launch
    float best = 0.f;
    cudaError_t e = cudaSuccess;
    for (int rep = 0; rep < 4 && e == cudaSuccess; ++rep) {
        e = cudaEventRecord(e0);
        if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, batch_peak_kernel, iters);
        if (e == cudaSuccess) e = cudaEventRecord(e1);
        if (e == cudaSuccess) e = cudaEventSynchronize(e1);
        float ms = 0.f;
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        if (e == cudaSuccess && rep > 0 && (best == 0.f || ms < best)) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (e != cudaSuccess) return fail(PBX_E_CUDA, "int8 peak measurement failed: %s", cudaGetErrorString(e));
    // per accumulator and CTA: 128 x 256 x 256 multiply-accumulates
    *out_tops = 2.0 * 128.0 * 256.0 * 256.0 * (double)iters * (double)sms / ((double)best * 1e-3) / 1e12;
    return PBX_OK;
}

extern "C" int pbx_get_stats(const pbx_corpus* cc, pbx_stats* out) {
    pbx_corpus* c = const_cast<pbx_corpus*>(cc);
    if (!c || !out) return fail(PBX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(c->mu);
    memset(out, 0, sizeof(*out));
    out->rows = c->n.load() + c->pending.load();
    out->capacity_rows = c->capacity.load();
    out->reserved = c->use_vmm ? 1 : 0;             // 1: the arrays grow by mapping memory into reserved address ranges
    out->dim = c->dim;
    out->row_pitch = c->pitch;
    out->queries = c->queries;
    unsigned long long xp = 0;
    CU_TRY(cudaSetDevice(c->device));
    CU_TRY(cudaMemcpy(&xp, c->d_exact_passes, sizeof(xp), cudaMemcpyDeviceToHost));
    out->exact_passes = xp;
    out->last_search_ms = c->last_search_ms;
    out->last_scan_ms = c->last_scan_ms;
    out->last_bytes_scanned = c->last_bytes;
    out->device = c->device;
    out->sm_count = c->sm_count;
    out->scan_grid = c->last_grid ? c->last_grid : scan_grid(c);
    out->batched_queries = c->batched_queries;
    return PBX_OK;
}

extern "C" int pbx_set_candidate_slack(pbx_corpus* c, uint32_t slack) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    c->slack = slack;
    return PBX_OK;
}

extern "C" int pbx_set_profiling(pbx_corpus* c, int enabled) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    c->profiling = enabled != 0;
    return PBX_OK;
}

extern "C" int pbx_set_batch_min(pbx_corpus* c, uint32_t min_queries) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    c->batch_min = min_queries ? min_queries : 2u;
    return PBX_OK;
}

extern "C" int pbx_set_scan_ctas_per_sm(pbx_corpus* c, uint32_t ctas_per_sm) {
    if (!c) return fail(PBX_E_INVALID, "corpus is NULL");
    if (ctas_per_sm > 8) return fail(PBX_E_INVALID, "ctas_per_sm must be <= 8");
    std::lock_guard<std::mutex> lk(c->mu);
    c->ctas_per_sm = ctas_per_sm;
    return PBX_OK;
}

#ifdef PBX_BATCH_PROF
// experiment builds only (not declared in the public header): per-CTA role counters of batch_mma_kernel
extern "C" __attribute__((visibility("default"))) int pbx_debug_batch_profile(unsigned long long* out, int reset) {
    if (out && cudaMemcpyFromSymbol(out, g_batch_prof, sizeof(unsigned long long) * 2048 * 12) != cudaSuccess) return -1;
    if (reset) {
        static unsigned long long zeros[2048 * 12];
        if (cudaMemcpyToSymbol(g_batch_prof, zeros, sizeof(zeros)) != cudaSuccess) return -1;
    }
    return 0;
}
#endif
#ifdef PBX_EXP_PROFILE
extern "C" __attribute__((visibility("default"))) int pbx_debug_fin_profile(long long* out) {
    return cudaMemcpyFromSymbol(out, g_fin_prof, sizeof(long long) * 16) == cudaSuccess ? 0 : -1;
}
// experiment builds only (not declared in the public header)
extern "C" __attribute__((visibility("default"))) int pbx_debug_scan_profile(unsigned long long* out, int reset) {
    if (out && cudaMemcpyFromSymbol(out, g_scan_prof, sizeof(unsigned long long) * kMaxScanGrid * 8) != cudaSuccess) return -1;
    if (reset) {
        static unsigned long long zeros[kMaxScanGrid * 8];
        if (cudaMemcpyToSymbol(g_scan_prof, zeros, sizeof(zeros)) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

#include "sharded.inl"
