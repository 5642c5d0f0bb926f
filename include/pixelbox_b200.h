/*
 * pixelbox_b200.h -- C ABI of the B200-native similarity-search library for PixelBox.
 *
 * This is the drop-in boundary for ONE path of the reference (JosephCatrambone/pixelbox): the
 * brute-force cosine-distance scan + top-k over the u8-quantized hashes of the SQLite
 * `semantic_hashes` table.  The reference has no FFI for this path today; each entry point
 * below names the reference code it replaces (paths relative to the reference checkout) and
 * INTEGRATION.md shows the Rust `extern "C"` block and the engine.rs patch that binds them.
 *
 * Conventions
 *   - plain C, no C++ types, no exceptions across the boundary; every call returns PBX_OK (0)
 *     or a negative PBX_E_* code; pbx_last_error() gives a thread-local message.
 *   - the caller owns every input and output buffer; the library copies inputs before it returns.
 *   - a pbx_corpus is one device-resident shard of the table on ONE B200 (sm_100).  There is
 *     no CPU fallback: without an sm_100 device pbx_corpus_create fails with PBX_E_NO_DEVICE.
 *   - results are the reference's: rows with (f64)dist < max_dist, ordered by (dist asc,
 *     image_id asc), at most k of them (src/engine.rs:379-381), where dist is the reference's
 *     f32 cosine_distance (src/engine.rs:572-588) reproduced bit for bit.
 */
#ifndef PIXELBOX_B200_H
#define PIXELBOX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define PBX_API __declspec(dllexport)
#else
#define PBX_API __attribute__((visibility("default")))
#endif

#define PBX_OK 0
#define PBX_E_INVALID (-1)     /* null pointer, k == 0 where not allowed, bad sizes            */
#define PBX_E_DIM (-2)         /* dim == 0 or dim > PBX_MAX_DIM                                  */
#define PBX_E_OOM (-3)         /* host or device allocation failed                              */
#define PBX_E_CUDA (-4)        /* a CUDA runtime call or kernel failed                          */
#define PBX_E_NO_DEVICE (-5)   /* no sm_100 (B200) device: there is no CPU fallback             */
#define PBX_E_CAPACITY (-6)    /* more than PBX_MAX_ROWS rows in one shard                      */
#define PBX_E_K (-7)           /* k > PBX_MAX_K                                                  */
#define PBX_E_INTERNAL (-8)    /* an internal invariant failed (a bug; never a silent wrong answer) */

#define PBX_MAX_DIM 4096u
#define PBX_MAX_K 2048u
#define PBX_MAX_ROWS 0xFFFFF000ull   /* capacity rounding and the +1023 terms of the kernels stay inside 32 bits */
#define PBX_MAX_SHARDS 64u

/* Per-query error markers in the count output of the device-resident calls (pbx_search_device,
 * pbx_exchange_allgather_merge); valid counts are <= k <= PBX_MAX_K.  The host-buffer calls never return them: they
 * repair the query (exact pass re-run from the host) or fail with PBX_E_INTERNAL. */
#define PBX_COUNT_EXCHANGE_TIMEOUT 0xFFFFFFFFu    /* a peer did not post its records within ~10 s               */
#define PBX_COUNT_EXACT_LAUNCH_FAILED 0xFFFFFFFEu /* the device-side launch of the exact pass was refused: the  */
                                                  /* hits of this query are the uncertified fast-pass ones      */
#define PBX_COUNT_FILTER_UNSORTED 0xFFFFFFFDu     /* pbx_search_device_filtered: the filter ids were not sorted */
                                                  /* ascending; the hits of every query of the call are invalid */

/* Filter modes of the *_filtered searches. */
#define PBX_FILTER_INCLUDE 0u   /* only rows whose image_id is listed      */
#define PBX_FILTER_EXCLUDE 1u   /* every row except those whose id is listed */

/* DEFAULT_MAX_QUERY_DISTANCE and the literal LIMIT of the reference (src/engine.rs:23, :381). */
#define PBX_DEFAULT_MAX_DIST 1e3
#define PBX_DEFAULT_K 100u

typedef struct pbx_corpus pbx_corpus;

/* One result row.  image_id / dist are what src/engine.rs:384-387 reads back from SQLite
 * (row.get(0), row.get(7)); dot / norm2 are the exact integer terms of SURVEY.md section 8a:
 * dot = sum c(q_i) c(r_i), norm2 = sum c(r_i)^2 with c(v) = 2v - 255.
 * Also the record the shards exchange (one NCCL all-gather of k of these per query). */
typedef struct pbx_hit {
    int64_t image_id;
    float dist;
    int32_t dot;
    int32_t norm2;
    uint32_t flags; /* bit 0: produced by the exact (tie-resolving) pass */
} pbx_hit;

typedef struct pbx_stats {
    uint64_t rows;             /* committed rows                                   */
    uint64_t capacity_rows;    /* allocated rows                                   */
    uint32_t dim;
    uint32_t row_pitch;        /* bytes between rows in HBM (dim rounded up to 16) */
    uint64_t queries;          /* queries answered since create                    */
    uint64_t exact_passes;     /* queries that needed the exact tie-resolving pass */
    float last_search_ms;      /* device time of the last pbx_search (CUDA events); needs pbx_set_profiling */
    float last_scan_ms;        /* ... of the scan kernel of its last query; needs pbx_set_profiling        */
    uint64_t last_bytes_scanned; /* rows * dim * nq of the last pbx_search         */
    int32_t device;
    int32_t sm_count;
    int32_t scan_grid;         /* CTAs of the persistent scan kernel               */
    int32_t reserved;          /* 1: the shard grows by mapping memory into reserved address ranges (no copy) */
    uint64_t batched_queries;  /* queries answered by the tensor-core batched path */
} pbx_stats;

/* ---- lifecycle -------------------------------------------------------------------------
 * Replaces: the table itself, `CREATE TABLE semantic_hashes (image_id INTEGER PRIMARY KEY,
 * hash BLOB)` (src/engine.rs:48, :109), as the thing the scan reads.  `device` is a CUDA
 * ordinal; capacity_hint rows are reserved up front (the corpus still grows on append). */
PBX_API int pbx_corpus_create(uint32_t dim, uint64_t capacity_hint, int device, pbx_corpus** out);
PBX_API void pbx_corpus_destroy(pbx_corpus* c);

/* Replaces: nothing upstream does this explicitly -- SQLite pages the table in during every
 * scan.  Hook: Engine::open after src/engine.rs:129, fed by
 * `SELECT image_id, hash FROM semantic_hashes ORDER BY image_id`.  Discards previous contents.
 * hashes is [n][dim] row-major u8.  Rows whose blob length != dim cannot be expressed here;
 * the caller must reject them (the reference would zip-truncate, src/engine.rs:585). */
PBX_API int pbx_corpus_load(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n);

/* Replaces: the hash INSERT of src/engine.rs:251-256 as seen by later scans.  Hook: the writer
 * loop src/engine.rs:188-200, after the INSERT reports a changed row.  Safe to call while
 * another thread is inside pbx_search: a search sees a committed prefix of the rows. */
PBX_API int pbx_corpus_append(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n);
/* Appends of fewer than 64 rows are collected on the host and uploaded 1024 at a time (the writer loop inserts one image
 * at a time); they count as part of the table at once: pbx_corpus_size includes them and every search uploads them before
 * it runs.  pbx_corpus_flush uploads them now.  An append that would take the shard (pending rows included) past
 * PBX_MAX_ROWS rows, or past the rows its address range was reserved for, returns PBX_E_CAPACITY and changes nothing,
 * coalesced or not.  The shard grows by mapping more device memory behind its arrays (CUDA
 * virtual memory management): no copy, no moved pointer, searches keep running while it grows. */
PBX_API int pbx_corpus_flush(pbx_corpus* c);
/* The same for rows that are already in device memory on the corpus' device (e.g. produced by pbx_quantize_device):
 * d_hashes is [n][dim] u8, d_image_ids [n] i64, both DEVICE pointers; the copy and the metadata kernels run on
 * `cuda_stream` (a cudaStream_t; NULL = an internal stream), which is synchronised before the rows are published. */
PBX_API int pbx_corpus_append_device(pbx_corpus* c, const int64_t* d_image_ids, const uint8_t* d_hashes, uint64_t n, void* cuda_stream);

/* Replaces: `DELETE FROM semantic_hashes WHERE image_id IN (...)` as seen by later scans.  Hook: after the DELETE of a
 * removed tracked folder commits (the TODO of remove_tracked_folder, src/engine.rs:414), with the folder's image ids; also
 * what follows an external edit of the table.  To replace a hash, use pbx_corpus_replace: a remove then an append is
 * not atomic (a search in between misses the image) and moves rows.
 *   - every committed or pending row whose image_id is in image_ids[0, n) is removed; the corpus does not enforce unique
 *     ids, so an id on several rows removes all of them.  Ids that match nothing are ignored; an id repeated in the
 *     request counts once.  *out_removed (may be NULL) receives the number of rows removed.
 *   - n == 0 returns PBX_OK with 0 removed; NULL c, or NULL image_ids with n > 0, is PBX_E_INVALID.
 *   - synchronous, and atomic with respect to searches: a search sees all of a removal or none of it.  Work already
 *     enqueued by pbx_search_device (on any stream) completes against the old rows; every search issued after the call
 *     returns gives exactly what a corpus freshly loaded with the surviving rows gives (ids, dist bit for bit, dot, norm2).
 *   - appends that arrived before the call (coalesced pending ones included) are subject to it, later ones are not: remove
 *     then append of the same id replaces the row.
 *   - capacity is not released; later appends reuse the freed rows.  Surviving rows may change position: the removed
 *     rows below the new size n' are filled, in row order, with the surviving rows at or above n', in row order.
 * Cost: a host sort of the request, one pass over the ids (8 bytes per row) plus the block metadata (8 bytes per row) on
 * the device, and a copy of the moved rows only. */
PBX_API int pbx_corpus_remove(pbx_corpus* c, const int64_t* image_ids, uint64_t n, uint64_t* out_removed);

/* Replaces: `UPDATE semantic_hashes SET hash = ? WHERE image_id = ?` as seen by later scans, one statement per listed id,
 * in order.  Hook: after such an UPDATE commits (a re-index of a modified file, a re-hash after a model fix, an external
 * edit of the table).  hashes is [n][dim] row-major u8: hashes[i] is the new hash of image_ids[i].
 *   - every committed or pending row whose image_id is listed gets the hash listed for that id, in place: positions, ids
 *     and the size do not change (pbx_corpus_read_rows shows the new bytes at the same positions).  An id on several
 *     rows replaces all of them; an id listed more than once takes its LAST hash; ids that match nothing are ignored.
 *   - *out_replaced (may be NULL) receives the number of rows written, counted as SQLite's changes(): a row counts even
 *     when its new hash equals the old one.
 *   - n == 0 returns PBX_OK; NULL c, NULL image_ids or hashes with n > 0, or n > PBX_MAX_ROWS is PBX_E_INVALID.
 *   - synchronous, and atomic with respect to searches, as pbx_corpus_remove: appends that arrived before the call
 *     (coalesced pending ones included) are subject to it; work already enqueued by pbx_search_device (on any stream)
 *     completes against the old hashes; every search issued after the call returns gives exactly what a corpus freshly
 *     loaded with the updated table, in the same row order, gives (ids, dist bit for bit, dot, norm2).
 * Cost: a host sort of the request (skipped for ids already strictly ascending) and its upload, one pass over the ids
 * (8 bytes per row) on the device, and a copy plus the row and 32-row-block metadata of the written rows only. */
PBX_API int pbx_corpus_replace(pbx_corpus* c, const int64_t* image_ids, const uint8_t* hashes, uint64_t n, uint64_t* out_replaced);

/* ---- views: a prepared id set, searched at the cost of its own rows ------------------------------------------------------
 * Replaces: the per-call filter of a search repeated over the same set -- "similar images in this folder", asked again and
 * again while the folder changes only when images are indexed into it or removed.  A filtered search streams the whole
 * shard every call; a search on a view streams the view's rows only.
 * A view is a pbx_corpus on the parent's device holding a copy of the parent's rows whose image_id is in a set of ids
 * (the INCLUDE semantics of the filtered searches: ids that match nothing are ignored, a repeated id counts once, an id on
 * several rows brings all of them).  Every search call accepts it (pbx_search, _hits, _device, _filtered, _page, their
 * device forms, pbx_exchange_search_hits*), and so do pbx_corpus_size / _read_rows / _synchronize / _flush, pbx_get_stats
 * and the pbx_set_* knobs.  pbx_corpus_load / _append / _append_device / _remove / _replace / _fill_synthetic on a view
 * return PBX_E_INVALID: a view follows its parent.  pbx_corpus_destroy destroys it.
 *   - Same results: a search on a view returns exactly what pbx_search_filtered (PBX_FILTER_INCLUDE, the view's set) returns
 *     on the parent at that moment -- count, ids, order, dist bit for bit, dot, norm2, and the plateau rule over the view's
 *     rows -- on every path: single, batched, paged, device forms, sharded and exchange.  The one difference: rows with
 *     equal (dist, image_id) may come in another order.  That needs an id on several rows, and a view's row order may
 *     differ from the parent's after removals.  A filter on a search of a view intersects with the view's set.
 *   - The view follows its parent inside the parent's mutating calls, which already hold the parent's locks and
 *     synchronise: appended rows (pbx_corpus_append, _append_device, coalesced appends when they are uploaded) whose id is
 *     in the set join the view; pbx_corpus_remove and pbx_corpus_replace are applied to the view as well (its rows, ids,
 *     row metadata stay the parent's bit for bit); pbx_corpus_load and _fill_synthetic rebuild it from the new rows.
 *     Removing a row does not take its id out of the set: a later append of that id joins the view, as it would pass the
 *     filter.  Each mutation and its forwarding are one step for searches on the view, as the remove and replace contracts
 *     say: work already enqueued on the view finishes against the old rows, every search issued after the call returns
 *     sees the new ones.
 *   - A search on a view first uploads the parent's pending appends (as a search of the parent does), and so do
 *     pbx_corpus_size, _read_rows and _flush on a view.
 *   - If the parent is destroyed first, its views are detached: they keep their rows and stay searchable;
 *     pbx_corpus_view_add on a detached view returns PBX_E_INVALID (pbx_corpus_view_drop still works).
 *   - NULL out_view / view / parent, NULL ids with n > 0, n > PBX_MAX_ROWS, a view of a view, or view_add / view_drop on a
 *     corpus that is not a view: PBX_E_INVALID.
 * Cost: m rows take m * (pitch + 16.5) bytes of device memory, allocated as a corpus' are (whole 2 MB pages per array under
 * CUDA virtual memory management), plus 8 bytes per id of the set on the device and on the host, plus the search scratch
 * every corpus has.  Building a view is a host sort of the ids, one mark pass over the parent's ids (8 bytes per row, a
 * binary search in the set per row) and a copy of the m rows on the device; pbx_corpus_view_add is the same over the ids
 * new to the set; view_drop is a pbx_corpus_remove on the view.  Each parent append adds, per view, a mark pass over the
 * appended rows and a copy of those that join; each parent remove or replace adds the same call on the view's m rows.
 * A search costs a search over m rows. */
PBX_API int pbx_corpus_view_create(pbx_corpus* parent, const int64_t* ids, uint64_t n, pbx_corpus** out_view);
/* The set grows or shrinks: rows of the parent with an added id join the view (*out_rows_added, may be NULL, counts them;
 * ids already in the set add nothing), rows with a dropped id leave it (*out_rows_dropped, may be NULL).  Atomic for
 * searches on the view, as pbx_corpus_remove. */
PBX_API int pbx_corpus_view_add(pbx_corpus* view, const int64_t* ids, uint64_t n, uint64_t* out_rows_added);
PBX_API int pbx_corpus_view_drop(pbx_corpus* view, const int64_t* ids, uint64_t n, uint64_t* out_rows_dropped);

/* Bench/test only: fills the shard on the device with rows [first_row, first_row + n) of the
 * counter-based synthetic corpus (pixelbox_b200/synth.py), image_id = global row + 1. */
PBX_API int pbx_corpus_fill_synthetic(pbx_corpus* c, uint64_t n, uint64_t seed, uint64_t first_row);

PBX_API int pbx_corpus_size(const pbx_corpus* c, uint64_t* n_rows);
PBX_API int pbx_corpus_dim(const pbx_corpus* c, uint32_t* dim);

/* Copies rows [first, first + n) back to the host (tests, and result hydration of
 * IndexedImage.visual_hash, src/engine.rs:385).  Either output may be NULL.  Row positions are those of the moment:
 * pbx_corpus_remove moves surviving rows into the positions of removed ones. */
PBX_API int pbx_corpus_read_rows(const pbx_corpus* c, uint64_t first, uint64_t n, int64_t* image_ids, uint8_t* hashes);

/* Waits for everything enqueued on the corpus' own stream (pbx_search_device with a NULL stream). */
PBX_API int pbx_corpus_synchronize(pbx_corpus* c);

/* ---- search ----------------------------------------------------------------------------
 * Replaces: the SQL statement of Engine::query_by_image_hash_from_image,
 *   SELECT ..., cosine_distance(?, semantic_hashes.hash) AS dist FROM semantic_hashes ...
 *   WHERE dist < ? ORDER BY dist ASC LIMIT 100            (src/engine.rs:375-383)
 * together with the scalar UDF it calls per row (src/engine.rs:608-622) and the distance
 * function itself (src/engine.rs:572-588).  queries is [nq][dim] u8 (IndexedImage.visual_hash,
 * src/indexed_image.rs:28); k replaces the literal LIMIT; max_dist is
 * Engine.max_distance_from_query (src/engine.rs:92), compared as `(f64)dist < max_dist`.
 * Outputs are [nq][k]; out_count[q] <= k rows are valid for query q; any of out_dist, out_dot,
 * out_norm2 may be NULL.  Synchronous: host buffers in, host buffers out. */
PBX_API int pbx_search(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                       int64_t* out_ids, float* out_dist, int32_t* out_dot, int32_t* out_norm2,
                       uint32_t* out_count);

/* Same search, but as the per-shard half of a row-sharded corpus: leaves [nq][k] pbx_hit
 * records (unused tail slots have image_id = INT64_MAX, dist = +inf) and [nq] counts in host
 * memory, ready for the all-gather. */
PBX_API int pbx_search_hits(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                            pbx_hit* out_hits, uint32_t* out_count);

/* Device-resident, asynchronous variant: d_queries [nq][dim], d_hits [nq][k] and d_count [nq]
 * are DEVICE pointers on the corpus' device; the work is enqueued on `cuda_stream` (a
 * cudaStream_t; NULL = the corpus' own stream) and the call returns without waiting.  This is
 * what a pipeline (or the multi-GPU driver, which all-gathers d_hits with NCCL on the same
 * stream) uses; no host synchronisation happens inside.
 * Stream-ordering contract: the first kernel of a call is launched with programmatic stream
 * serialisation and reads d_queries in its prologue.  d_queries must therefore be complete in
 * stream order in the ordinary sense: written by copies, by kernels that have finished, or by a
 * preceding kernel on `cuda_stream` that does NOT trigger its dependents early
 * (cudaTriggerProgrammaticLaunchCompletion / griddepcontrol.launch_dependents) before its last
 * write to d_queries.  The library's own kernels never trigger early. */
PBX_API int pbx_search_device(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist,
                              pbx_hit* d_hits, uint32_t* d_count, void* cuda_stream);

/* ---- filtered search: the k nearest rows among a set of image ids ----------------------------------------------------
 * Replaces: the similarity query with an id condition added,
 *   ... FROM semantic_hashes ... WHERE dist < ? AND semantic_hashes.image_id IN (...)      (PBX_FILTER_INCLUDE)
 *   ... FROM semantic_hashes ... WHERE dist < ? AND semantic_hashes.image_id NOT IN (...)  (PBX_FILTER_EXCLUDE)
 *   ORDER BY dist ASC LIMIT k
 * which the `similar:` term of Engine::query (src/engine.rs:282-292) meant to combine with filename and tag terms, and
 * which a folder search ("similar images in this folder") needs; the host turns such conditions into ids.
 *   - Each call takes the arguments of its unfiltered twin plus (filter_ids, n_filter, filter_mode).  One filter applies
 *     to all nq queries of the call.
 *   - Contract: the result is exactly what the unfiltered twin returns on a corpus loaded with only the allowed rows:
 *     count, ids, order, dist bit for bit, dot, norm2, ties by image_id, and the plateau rule applied to allowed rows.
 *   - The filter applies to the rows that exist when the call is made, coalesced pending appends included; rows that
 *     pbx_corpus_remove moved are found by id.  Ids that match no row are ignored, a repeated id counts once, and an id
 *     on several rows includes or excludes all of them.
 *   - An empty INCLUDE set gives count 0 for every query; an empty EXCLUDE set is the unfiltered search.
 *   - NULL filter_ids with n_filter > 0, an unknown filter_mode or n_filter > PBX_MAX_ROWS: PBX_E_INVALID.
 *   - Host forms accept the ids in any order (a sorted copy is made; ids already in order cost one check pass).
 * Cost: the unfiltered search (the whole shard is streamed, whatever the filter selects: a selective filter is not
 * faster) plus one mark pass over the row ids (8 bytes per row, a binary search in the set per row).  On the batched
 * path (many queries per call) a very selective filter costs several times the unfiltered call (DESIGN.md section 10). */
PBX_API int pbx_search_filtered(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                int64_t* out_ids, float* out_dist, int32_t* out_dot, int32_t* out_norm2, uint32_t* out_count,
                                const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode);
/* Device-resident form, with the contract of pbx_search_device.  d_filter_ids is a DEVICE pointer on the corpus' device,
 * read in stream order on `cuda_stream`; it must be sorted ascending (duplicates allowed).  The order is checked on the
 * device, without a host synchronisation: unsorted ids set every count of the call to PBX_COUNT_FILTER_UNSORTED. */
PBX_API int pbx_search_device_filtered(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist,
                                       pbx_hit* d_hits, uint32_t* d_count, void* cuda_stream,
                                       const int64_t* d_filter_ids, uint64_t n_filter, uint32_t filter_mode);

/* ---- paged search: the k rows after a (dist, image_id) cursor ----------------------------------------------------------
 * Replaces: keyset pagination of the similarity query ("show more", or more than PBX_MAX_K rows in all),
 *   ... FROM semantic_hashes ... WHERE dist < :max_dist AND (dist > :d0 OR (dist = :d0 AND image_id > :id0))
 *   [AND image_id IN / NOT IN (...)]  ORDER BY dist ASC, image_id ASC LIMIT k
 *   - Each call takes its twin's arguments plus the cursors and the filter triple of the *_filtered searches
 *     (n_filter = 0 with PBX_FILTER_EXCLUDE: unfiltered; same argument rules).  Outputs are pbx_hit records.
 *   - after[q] is query q's cursor: only its image_id (id0) and dist (d0) are read, so the next cursor is the last hit of
 *     the previous page.  after == NULL: the first page of every query.  {dist = -inf, image_id = INT64_MIN} is also "from
 *     the start" (no row sorts at or before it); dist = +inf gives count 0.  The cursor need not be a row of the table:
 *     any (d0, id0) works, an id that was removed or never existed included.
 *   - A NaN d0: PBX_E_INVALID on the host forms; on the device form that query gets count 0.
 *   - Contract: exactly the SQL above -- count, ids, order, dist bit for bit, dot, norm2, ties by image_id, and the plateau
 *     rule applied to the rows after the cursor.  The pages of one iteration concatenate to the first rows of one deep
 *     top-K for any K, past PBX_MAX_K included, with or without a filter.
 *   - Pages follow the table at the time of each call (nothing is stored between calls): a row appended between two calls
 *     shows up on a later page if it sorts after the cursor, and is never seen if it sorts before it.
 *   - Image ids need not be unique: rows with the same (dist, image_id) are all on the same side of a cursor, as in the SQL.
 * Cost: one search; a page at depth D adds about D candidate tests per query on the batched path (DESIGN.md section 10). */
PBX_API int pbx_search_page(pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist, const pbx_hit* after,
                            const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode, pbx_hit* out_hits, uint32_t* out_count);
/* Device-resident form, with the contract of pbx_search_device_filtered.  d_after [nq] (or NULL) is a DEVICE pointer on the
 * corpus' device, read in stream order on `cuda_stream` with no host read: a pipeline can pass the previous call's d_hits
 * (the record at slot count - 1 of each query) as the next cursors. */
PBX_API int pbx_search_device_page(pbx_corpus* c, const uint8_t* d_queries, uint32_t nq, uint32_t k, double max_dist,
                                   const pbx_hit* d_after, const int64_t* d_filter_ids, uint64_t n_filter, uint32_t filter_mode,
                                   pbx_hit* d_hits, uint32_t* d_count, void* cuda_stream);

/* ---- range search: every row within max_dist, and its exact count ------------------------------------------------------
 * Replaces: the similarity query without its LIMIT ("every copy of this photo", "everything inside max_distance"), and
 * its COUNT(*):
 *   SELECT image_id, cosine_distance(?, hash) AS dist FROM semantic_hashes WHERE dist < :max_dist
 *   [AND (dist > :d0 OR (dist = :d0 AND image_id > :id0))]  [AND image_id IN / NOT IN (...)]  ORDER BY dist ASC, image_id ASC
 *   - after (NULL or [nq] cursors) and the filter triple as in pbx_search_page (same argument rules; a NaN cursor dist is
 *     PBX_E_INVALID).  max_dist is compared as the f64 `dist < max_dist`: NaN gives no row; above 999999 every row is
 *     inside, the plateau rows ordered by image_id; a row at dist -1.19e-7 (an identical row) is inside even at max_dist 0.
 *   - out_total[q] is always the exact COUNT(*) of query q, whatever the capacity.
 *   - Rows are written query after query, each query's rows in order, until `capacity` rows are written: query q's rows
 *     are out_hits[out_offsets[q] .. out_offsets[q + 1]), a prefix of its answer (out_offsets has nq + 1 entries).  A query
 *     whose answer was cut continues with the same call and after = its last written row.
 *   - capacity = 0 counts only (out_hits may be NULL); NULL out_offsets / out_total, or NULL out_hits with capacity > 0,
 *     is PBX_E_INVALID.
 *   - Records carry dist bit for bit, dot and norm2, as the top-k records do (flags = 0).
 *   - Ordered like any search of the corpus (the previous search's kernels, pending appends uploaded first): a range
 *     search sees all of a removal or replacement or none of it.  A view (pbx_corpus_view_create) is searched like a corpus.
 * Cost: one streaming pass per query, plus the exact replay of the rows near max_dist (count only) or of the answer and a
 * sort that grows with it.  A host call: it reads the candidate count of each query once, and its result. */
PBX_API int pbx_search_range(pbx_corpus* c, const uint8_t* queries, uint32_t nq, double max_dist, const pbx_hit* after,
                             const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode, pbx_hit* out_hits, uint64_t capacity,
                             uint64_t* out_offsets, uint64_t* out_total);

/* Merge step after the all-gather (SURVEY.md section 8e): gathered is [n_shards][nq][k] hits and
 * counts is [n_shards][nq], both in HOST memory; every shard list is already ordered by
 * (dist, image_id).  Writes the global first k per query under the same order.  Pure host
 * logic (a k-way merge of <= n_shards*k records), usable without a GPU. */
PBX_API int pbx_merge_hits(const pbx_hit* gathered, const uint32_t* counts, uint32_t n_shards, uint32_t nq, uint32_t k,
                           pbx_hit* out_hits, uint32_t* out_count);

/* Device-side form of the same merge for pipelines that keep the gathered records in HBM (the
 * buffer an NCCL all-gather of the pbx_search_device outputs produces): all pointers are DEVICE
 * pointers; d_counts may be NULL, in which case each list's length is the number of leading slots
 * with a finite dist (so only the hit records need to be exchanged).  The kernel is enqueued on `cuda_stream` (NULL = the legacy default stream) of
 * `device` and the call does not wait. */
PBX_API int pbx_merge_hits_device(int device, const pbx_hit* d_gathered, const uint32_t* d_counts, uint32_t n_shards,
                                  uint32_t nq, uint32_t k, pbx_hit* d_out_hits, uint32_t* d_out_count, void* cuda_stream);

/* ---- the row-sharded corpus of ONE process over several GPUs -------------------------------------------------------
 * Replaces: the same table and query as pbx_corpus / pbx_search, for a corpus that needs more than one GPU (1B x 256 B =
 * 256 GB).  The reference's host is a single process that calls Engine on the UI thread (src/ui/search.rs:20-31,
 * src/engine.rs:117-145), so this is what its FFI crate binds when several devices are named.  `devices` lists CUDA
 * ordinals (repeats allowed: several shards on one GPU); rows are partitioned by contiguous blocks of the id-ordered
 * table at load, appended rows go to the emptiest shard; image ids stay global.  A search runs the complete local search
 * on every shard (one worker thread and stream per shard), copies each shard's k records per query to the first device
 * over NVLink and merges them there under (dist, image_id): results are identical to one pbx_corpus holding all rows. */
typedef struct pbx_sharded pbx_sharded;
PBX_API int pbx_sharded_create(uint32_t dim, uint64_t capacity_hint, const int* devices, int n_devices, pbx_sharded** out);
PBX_API void pbx_sharded_destroy(pbx_sharded* s);
PBX_API int pbx_sharded_load(pbx_sharded* s, const int64_t* image_ids, const uint8_t* hashes, uint64_t n);
PBX_API int pbx_sharded_append(pbx_sharded* s, const int64_t* image_ids, const uint8_t* hashes, uint64_t n);
/* pbx_corpus_remove over all shards: ids are global and do not name a shard, so every shard applies the whole request
 * (one after the other, atomic with respect to pbx_sharded_search); *out_removed (may be NULL) is the total. */
PBX_API int pbx_sharded_remove(pbx_sharded* s, const int64_t* image_ids, uint64_t n, uint64_t* out_removed);
/* pbx_corpus_replace over all shards, in the same way: every shard applies the whole request (one after the other,
 * atomic with respect to pbx_sharded_search); *out_replaced (may be NULL) is the total. */
PBX_API int pbx_sharded_replace(pbx_sharded* s, const int64_t* image_ids, const uint8_t* hashes, uint64_t n, uint64_t* out_replaced);
/* Views over a pbx_sharded: one view per shard, each of its own shard (ids are global), with pbx_corpus_view_create's
 * contract.  Every pbx_sharded_search* accepts the result; pbx_sharded_load / _append / _remove / _replace /
 * _fill_synthetic on it return PBX_E_INVALID; pbx_sharded_destroy destroys it.  The outputs of _add / _drop are totals. */
PBX_API int pbx_sharded_view_create(pbx_sharded* parent, const int64_t* ids, uint64_t n, pbx_sharded** out_view);
PBX_API int pbx_sharded_view_add(pbx_sharded* view, const int64_t* ids, uint64_t n, uint64_t* out_rows_added);
PBX_API int pbx_sharded_view_drop(pbx_sharded* view, const int64_t* ids, uint64_t n, uint64_t* out_rows_dropped);
/* Bench/test only: shard i holds rows [i * rows_per_shard, (i + 1) * rows_per_shard) of the synthetic corpus. */
PBX_API int pbx_sharded_fill_synthetic(pbx_sharded* s, uint64_t rows_per_shard, uint64_t seed);
PBX_API int pbx_sharded_size(const pbx_sharded* s, uint64_t* n_rows);
PBX_API int pbx_sharded_shards(const pbx_sharded* s, uint32_t* n_shards);
/* The i-th shard, for pbx_get_stats / the pbx_set_* knobs; owned by the sharded corpus. */
PBX_API int pbx_sharded_shard(pbx_sharded* s, uint32_t index, pbx_corpus** out);
/* Same contracts as pbx_search / pbx_search_hits (host buffers in, host buffers out, synchronous). */
PBX_API int pbx_sharded_search(pbx_sharded* s, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                               int64_t* out_ids, float* out_dist, int32_t* out_dot, int32_t* out_norm2, uint32_t* out_count);
PBX_API int pbx_sharded_search_hits(pbx_sharded* s, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                    pbx_hit* out_hits, uint32_t* out_count);
/* pbx_search_filtered over all shards: ids are global, every shard marks its rows against the same set; the merge is
 * unchanged (each shard's list is exact for its allowed rows, so the merged list is exact for all of them). */
PBX_API int pbx_sharded_search_filtered(pbx_sharded* s, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                        int64_t* out_ids, float* out_dist, int32_t* out_dot, int32_t* out_norm2, uint32_t* out_count,
                                        const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode);
/* pbx_search_page over all shards: every shard applies the same global cursor; the merge is unchanged (the global next k
 * rows after a cursor are the first k of the union of every shard's next k rows after it). */
PBX_API int pbx_sharded_search_page(pbx_sharded* s, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                    const pbx_hit* after, const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode,
                                    pbx_hit* out_hits, uint32_t* out_count);
/* pbx_search_range over all shards, same arguments and contract: every shard runs the range search of its rows, the root
 * device gathers each shard's first min(total, capacity) rows and orders them; the totals are summed. */
PBX_API int pbx_sharded_search_range(pbx_sharded* s, const uint8_t* queries, uint32_t nq, double max_dist, const pbx_hit* after,
                                     const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode, pbx_hit* out_hits,
                                     uint64_t capacity, uint64_t* out_offsets, uint64_t* out_total);

/* ---- the exchange step over NVLink peer memory (one process per GPU) ---------------------------------
 * Replaces: nothing upstream (PixelBox is single-process); it is the one exchange step of the row-sharded path
 * (SURVEY.md section 8e).  Each rank creates an exchange (a device mailbox for [world][nq][k] records, double
 * buffered, plus sequence flags), publishes its 64-byte CUDA IPC handle, receives everybody's handles by whatever
 * means the host has (the Python driver all-gathers them with torch.distributed once) and connects.  After that
 * pbx_exchange_allgather_merge is ONE kernel on `cuda_stream`: it writes this rank's d_local hits ([nq][k], as left
 * by pbx_search_device) into every peer's mailbox, signals, waits for all peers' records of the same call and merges
 * them under (dist, image_id) into d_out / d_out_count.  All ranks must make the same sequence of calls with the
 * same nq and k.  nq * k <= max_records and nq <= max_queries. */
typedef struct pbx_exchange pbx_exchange;
PBX_API int pbx_exchange_create(int device, uint32_t rank, uint32_t world, uint32_t max_records, uint32_t max_queries,
                                pbx_exchange** out);
PBX_API int pbx_exchange_handle(pbx_exchange* x, void* out_handle_64_bytes);
PBX_API int pbx_exchange_connect(pbx_exchange* x, const void* all_handles /* [world][64] */);
PBX_API int pbx_exchange_allgather_merge(pbx_exchange* x, const pbx_hit* d_local, uint32_t nq, uint32_t k, pbx_hit* d_out,
                                         uint32_t* d_out_count, void* cuda_stream);
/* The whole per-rank step with host buffers (what pbx_search_hits is for one GPU): H2D of the queries, this shard's
 * search, the exchange + merge kernel, D2H of the merged records, one synchronisation.  Every rank calls it with the same
 * queries and receives the global result.  nq <= 1024 per call. */
PBX_API int pbx_exchange_search_hits(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k, double max_dist,
                                     pbx_hit* out_hits, uint32_t* out_count);
/* The same step for a filtered search (pbx_search_filtered's filter contract): every rank passes the same global ids. */
PBX_API int pbx_exchange_search_hits_filtered(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k,
                                              double max_dist, pbx_hit* out_hits, uint32_t* out_count,
                                              const int64_t* filter_ids, uint64_t n_filter, uint32_t filter_mode);
/* The same step for a paged search (pbx_search_page's contract): every rank passes the same cursors and filter. */
PBX_API int pbx_exchange_search_hits_page(pbx_exchange* x, pbx_corpus* c, const uint8_t* queries, uint32_t nq, uint32_t k,
                                          double max_dist, const pbx_hit* after, const int64_t* filter_ids, uint64_t n_filter,
                                          uint32_t filter_mode, pbx_hit* out_hits, uint32_t* out_count);
PBX_API void pbx_exchange_destroy(pbx_exchange* x);

/* ---- the scalar function, for external users of the DB -----------------------------------
 * Replaces: `pub fn cosine_distance(&Vec<u8>, &Vec<u8>) -> f32` (src/engine.rs:572-588) for a
 * batch of pairs: a and b are [n][dim] u8 in host memory; out_dist[n] receives the reference's
 * f32 value bit for bit, out_dot / out_norm2_a / out_norm2_b (optional) the exact integers.
 * Runs on the GPU of `device`. */
PBX_API int pbx_cosine_distance_pairs(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim,
                                      float* out_dist, int32_t* out_dot, int32_t* out_norm2_a, int32_t* out_norm2_b);

/* ---- the other two registered scalar functions (SURVEY.md 8f N4) ---------------------------------
 * Replace, for a batch of pairs in host memory (a and b are [n][dim] u8):
 *   `pub fn byte_distance(&Vec<u8>, &Vec<u8>) -> f32`     src/engine.rs:590-592  (UDF registered at :624-638)
 *       out_dist = sum |a_i - b_i| / (255 * dim), bit for bit; out_l1 (optional) = the integer sum.
 *   `pub fn hamming_distance(&Vec<u8>, &Vec<u8>) -> f32`  src/engine.rs:594-604  (UDF registered at :640-654)
 *       upstream adds the per-byte bit counts in a u8: past 255 differing bits the sum wraps (release build; a
 *       debug build panics).  out_dist reproduces the wrapped value, (bits mod 256) / (8 * dim); out_bits
 *       (optional) = the true number of differing bits.  Upstream KATs: test_hamming_distance, :693-701.
 * No query upstream uses either function; they exist for external users of the database, like
 * pbx_cosine_distance_pairs.  n <= 2^26 pairs per call. */
PBX_API int pbx_byte_distance_pairs(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim,
                                    float* out_dist, uint32_t* out_l1);
PBX_API int pbx_hamming_distance_pairs(int device, const uint8_t* a, const uint8_t* b, uint64_t n, uint32_t dim,
                                       float* out_dist, uint32_t* out_bits);

/* ---- the ingest quantizer ---------------------------------------------------------------------
 * Replaces: the f32 -> u8 map of mlhash, `128u8.saturating_add_signed((f*128.0).max(-128.0).min(128.0) as i8)`
 * (src/image_hashes/efficientnet.rs:39; README.md:54 example [-1, 1, 0, 0.1] -> [0x00, 0xFF, 0x80, 0x8C]), for a batch
 * of n floats in host memory, so embeddings produced elsewhere can be appended in the table's encoding. */
PBX_API int pbx_quantize(int device, const float* embeddings, uint64_t n, uint8_t* out);
/* Device-resident, asynchronous form: both pointers are DEVICE pointers on `device`, the kernel is enqueued on
 * `cuda_stream` (NULL = the legacy default stream) and the call does not wait -- embeddings produced on the GPU go to
 * pbx_corpus_append_device without touching the host (src/image_hashes/efficientnet.rs:35-40). */
PBX_API int pbx_quantize_device(int device, const float* d_embeddings, uint64_t n, uint8_t* d_out, void* cuda_stream);

/* ---- diagnostics ------------------------------------------------------------------------- */
PBX_API int pbx_get_stats(const pbx_corpus* c, pbx_stats* out);
/* Tuning knob for tests: candidate slack of the fast pass (candidates = k + slack); 0 restores
 * the default.  A tiny slack forces the exact pass and must not change any result. */
PBX_API int pbx_set_candidate_slack(pbx_corpus* c, uint32_t slack);
/* Profiling: when enabled, pbx_search / pbx_search_hits record CUDA events around the whole search and around the
 * scan kernel of its last query (pbx_stats.last_search_ms / last_scan_ms).  Off by default: an event between two
 * kernels serialises launches that otherwise overlap (programmatic dependent launch). */
PBX_API int pbx_set_profiling(pbx_corpus* c, int enabled);
/* Calls with at least `min_queries` queries take the tensor-core path (tcgen05 kind::i8 contraction with the top-k
 * fused into the epilogue) when the shape allows it (row pitch a multiple of 32 bytes, <= 1024; enough rows to seed the
 * thresholds); fewer queries, or other shapes, loop over the single-query scan.  0 restores the default (2: one
 * streaming pass over the corpus serves all queries of the call, 2 to 128 queries cost ~1.15x one); UINT32_MAX disables the
 * batched path.  Results are identical either way. */
PBX_API int pbx_set_batch_min(pbx_corpus* c, uint32_t min_queries);
/* CTAs per SM of the persistent scan kernel (0 = default). */
PBX_API int pbx_set_scan_ctas_per_sm(pbx_corpus* c, uint32_t ctas_per_sm);
/* Measures the int8 tensor-pipe ceiling of `device` for the batched path's MMA shape (tcgen05.mma.cta_group::2.kind::i8,
 * 256 x 256 x 32 per instruction, operands resident in shared memory, accumulators never read): dense int8 TOP/s, best of
 * three ~10 ms launches.  This is the measured denominator of the batched path's roofline (bench.py); the nominal
 * figure is 4500. */
PBX_API int pbx_int8_peak(int device, double* out_tops);
PBX_API const char* pbx_last_error(void);
PBX_API const char* pbx_version(void);
PBX_API int pbx_device_count(void); /* number of sm_100 devices visible; 0 if none */

#ifdef __cplusplus
}
#endif
#endif /* PIXELBOX_B200_H */
