/*
 * svsb200.h -- C ABI of the B200-native retrieve engine behind svs.KB.retrieve / svs.AsyncKB.retrieve.
 *
 * The reference (Rhobota/svs 0.7.4) is pure Python and has no FFI for this path; the seam is the
 * private class `_EmbeddingsMatrix` (src/svs/kb.py:856-893) and the `superheavy()` closures
 * (src/svs/kb.py:1184-1189 async, 1622-1627 sync).  Every entry point below names the reference
 * code it replaces.  INTEGRATION.md shows the ctypes binding and the ~20-line patch to kb.py.
 *
 * Conventions
 *   - every call returns 0 on success or a negative SVSB_E_* code; nothing throws or aborts;
 *     svsb_last_error() returns a thread-local message for the last failing call on this thread;
 *   - there is NO CPU fallback: without a usable CUDA device svsb_create fails;
 *   - host pointers are plain caller-owned buffers; the library copies before returning;
 *   - svsb_query* may be called concurrently from several OS threads (AsyncKB runs the compute in
 *     the default thread pool without holding the KB lock, src/svs/kb.py:1180,1190);
 *     svsb_invalidate / svsb_load_* may race with in-flight queries: a query keeps the generation
 *     it started on alive until it returns (the reference relies on NumPy refcounts for the same).
 *   - k is clipped to the row count (src/svs/util.py:198-199) for every k, on one device or several; callers with a
 *     wider integer type clip BEFORE the int32 argument (svs_b200/engine.py: clamp_k);
 *   - +0.0 and -0.0 are different keys: +0.0 sorts before -0.0 (the reference's float comparison treats them as equal
 *     and orders them by index); harmless under the tolerance clause, stated here for completeness;
 *   - result order: score descending, ties by ascending row (== ascending embeddings.id for a rowid
 *     scan, src/svs/kb.py:603-609).  The reference's get_top_k orders exact ties by DEscending index
 *     (src/svs/util.py:203); BASELINE.json's north star prescribes ascending id.
 */
#ifndef SVSB200_H
#define SVSB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct svsb_engine svsb_t;

enum {
    SVSB_OK            = 0,
    SVSB_E_INVALID     = -1,   /* bad argument */
    SVSB_E_CUDA        = -2,   /* CUDA runtime error (message has the detail) */
    SVSB_E_NOT_LOADED  = -3,   /* query with no matrix resident (Python re-loads, as kb.py:866-877) */
    SVSB_E_SHAPE       = -4,   /* query d != matrix d, or empty matrix: Python raises ValueError, as np.dot does */
    SVSB_E_STATE       = -5,   /* load_rows/load_end without load_begin, too many rows, ... */
    SVSB_E_NOMEM       = -6,
    SVSB_E_NO_DEVICE   = -7    /* no CUDA device: there is no CPU path */
};

/* Normalisation policy of the load path (SURVEY.md section 8, hazard H1). */
enum {
    SVSB_NORM_CHECK     = 0,   /* compute row norms on the device, keep rows verbatim (default: the
                                  reference scores raw dot products, src/svs/kb.py:1623) */
    SVSB_NORM_NORMALIZE = 1    /* divide every row by its L2 norm on the device */
};

/* ---- lifetime: KB.__init__ ... KB.close()  (src/svs/kb.py:1420, 1455) -------------------------- */

/* device_ids == NULL / n_dev <= 0: use device 0.  With n_dev > 1 the matrix is row-sharded over the
 * devices in scan order and every query gathers the per-device top-k lists (SURVEY.md section 8e). */
int  svsb_create(const int* device_ids, int n_dev, svsb_t** out);
void svsb_destroy(svsb_t* e);

/* ---- load path: replaces _Querier.build_embeddings_matrix (src/svs/kb.py:573-618) and the cache
 *      fill of _EmbeddingsMatrix.get_sync / get (src/svs/kb.py:866-893) ------------------------ */

/* Start building a new generation of n rows x d float32.  n == 0 is legal (empty table, kb.py:595-601). */
int svsb_load_begin(svsb_t* e, int64_t n, int32_t d, int32_t norm_mode);
/* Append `count` rows (row-major, d floats each, little-endian f32 exactly as the SQLite blobs hold
 * them, src/svs/embeddings/util.py:15-23) and their embeddings.id values, in scan order.  Data is
 * staged through the engine's pinned ring and copied to the device asynchronously. */
int svsb_load_rows(svsb_t* e, const float* rows, const int64_t* emb_ids, int64_t count);
/* Zero-copy variant: borrow a pinned staging slab, fill rows/ids in place, commit `count` rows. */
int svsb_load_acquire_slab(svsb_t* e, float** rows, int64_t** emb_ids, int64_t* capacity_rows);
int svsb_load_commit_slab(svsb_t* e, int64_t count);
/* Finish: wait for the copies, run the row-norm kernel, publish atomically.  Fails with
 * SVSB_E_STATE if fewer/more than n rows were supplied (the reference asserts, kb.py:616). */
int svsb_load_end(svsb_t* e, uint64_t* generation);
/* The whole of build_embeddings_matrix (src/svs/kb.py:573-618) natively: scan the `embeddings` table (kb.py:80-83) of the
 * SQLite file at `path` in rowid order -- the reference's scan order, kb.py:603-609 -- on private READ-ONLY connections
 * (libsqlite3.so.0 bound at run time; `threads` connections scan contiguous rowid ranges in parallel, 0 = default),
 * blobs copied verbatim (float32 little-endian, src/svs/embeddings/util.py:15-23) through pinned slabs to their final
 * rows on the device(s), then the row-norm kernel, then atomic publication.  The reference's checks are kept: every blob
 * has the first row's length (kb.py:613), the row count matches COUNT(*) (kb.py:616).  Call it where the reference
 * rebuilds -- inside the KB's transaction, when its connection has nothing uncommitted.  SVSB_E_STATE: no libsqlite3,
 * cannot open the file (":memory:"), ragged rows ...: the caller falls back to svsb_load_begin / _rows / _end. */
int svsb_load_sqlite(svsb_t* e, const char* path, int32_t norm_mode, int32_t threads, uint64_t* generation, int64_t* n_out,
                     int32_t* d_out);
/* 1 if libsqlite3 could be bound. */
int svsb_sqlite_available(void);
/* The same scan into host arrays (no device involved): rows[capacity_rows][d] and/or emb_ids[capacity_rows] (either may
 * be NULL; both NULL just reports the shape).  d_expected >= 0 must match the table's row length. */
int svsb_sqlite_read(const char* path, int32_t threads, float* rows, int64_t* emb_ids, int64_t capacity_rows, int32_t d_expected,
                     int64_t* n_out, int32_t* d_out);
/* Abandon a load in progress (the resident generation, if any, is untouched). */
int svsb_load_abort(svsb_t* e);
/* Bench/test support: fill n x d on the device(s) from the counter-based generator
 * (oracle/svs_oracle.py: counter_uniform_rows), emb_id of row r = id0 + r * id_step, then normalise. */
int svsb_load_synthetic(svsb_t* e, int64_t n, int32_t d, uint64_t seed, int64_t id0, int64_t id_step,
                        uint64_t* generation);

/* ---- incremental update: instead of the full invalidate + rebuild the reference does after every bulk add / delete
 *      (src/svs/kb.py:1062, 1086, 1523, 1541; SURVEY.md section 8f rank 4) ------------------------------------------
 * Applies ONE committed batch of mutations of the `embeddings` table to the resident generation and publishes the
 * result as a new generation that SHARES the matrix buffers with the old one (queries in flight on the old generation,
 * and snapshots, are undisturbed -- what NumPy refcounts give the reference):
 *   del_ids[n_del]            embeddings.id of deleted rows (`DELETE FROM embeddings WHERE id = ?`, kb.py:403, 548): each
 *                             must be a live row; it is tombstoned (its key sorts below every live row's);
 *   add_rows[n_add][d], add_ids[n_add]
 *                             inserted rows (`INSERT INTO embeddings`, kb.py:310, 557), in insertion order; ids must be
 *                             ascending and greater than every live id -- what SQLite's rowid allocation guarantees --
 *                             so that appending them keeps "row order == scan order of a fresh rebuild" (kb.py:603-609).
 *                             Rows are appended behind the last row (the last shard of a multi-device engine); the
 *                             buffer grows geometrically (one device-to-device copy) when it is full.
 * Deletes are applied first (an id deleted and re-inserted in one transaction is a tombstone plus an append).
 * SVSB_E_STATE: no generation resident, a del id that is not live, ids not ascending, d mismatch, or the resident
 * generation was replaced while the update was being built -- nothing is published and the caller falls back to the full
 * rebuild.  One update at a time (serialised inside); do not run it concurrently with svsb_load_begin .. svsb_load_end.  The result equals a fresh rebuild bit for bit: same ids,
 * same scores (tests/test_gpu_mutate.py).  Generations with tombstones answer batches and large k through the exact
 * kernels; svsb_top_pairs asks for a reload (SVSB_E_INVALID), on one device or several. */
int svsb_apply_mutations(svsb_t* e, const int64_t* del_ids, int64_t n_del, const float* add_rows, const int64_t* add_ids,
                         int64_t n_add, int32_t d, uint64_t* generation);
/* Physical rows of the resident generation (tombstoned ones included) and live rows (== svsb_shape's n). */
int svsb_generation_rows(svsb_t* e, int64_t* physical, int64_t* live);

/* The same update for one rank of the one-process-per-GPU deployment, in two phases, so that no rank publishes unless
 * every rank can.  Every rank calls both with the same arguments (SPMD); this engine owns one device.
 *   svsb_shard_mutations_prepare  builds the next generation of this rank's shard off to the side and keeps it pending in
 *                            the engine; nothing is published.  A delete id that is not a live row of THIS shard is not an
 *                            error: *found counts the ones that were.  *max_live_id: this shard's largest live id after
 *                            the deletes (INT64_MIN: none).  Only the rank with append_here != 0 (the last rank) appends
 *                            the rows, and it does everything that can fail there: buffer growth, row copy, norm kernel,
 *                            shadows.  Preconditions as svsb_apply_mutations (ids ascending, d, no duplicate delete ids,
 *                            2^32 rows counted from svsb_set_shard's offset); SVSB_E_STATE also while another update is
 *                            pending or a load runs.  The caller accepts the update only if every rank succeeded, the
 *                            found counts add up to n_del and add_ids[0] is above every rank's max_live_id.
 *   svsb_shard_mutations_commit   publish != 0 publishes the pending generation, 0 drops it (a no-op when nothing is
 *                            pending).  It allocates nothing and cannot fail after a successful prepare.
 * A pending generation blocks loads, updates and svsb_compact until it is committed or dropped; svsb_invalidate and
 * svsb_destroy drop it. */
int svsb_shard_mutations_prepare(svsb_t* e, const int64_t* del_ids, int64_t n_del, const float* add_rows, const int64_t* add_ids,
                                 int64_t n_add, int32_t d, int32_t append_here, int64_t* found, int64_t* max_live_id);
int svsb_shard_mutations_commit(svsb_t* e, int32_t publish, uint64_t* generation);
/* Compaction on the device (single-device engines; a multi-device engine gets SVSB_E_INVALID): gathers the live rows of
 * the resident generation, in row order, into a new buffer and publishes them as a tombstone-free generation whose first
 * row is global row global_row0 (svsb_set_shard's offset is set to it in the same call).  The result equals a fresh load
 * of the live rows at that offset: rows, ids, shape, svsb_norm_stats in check mode (normalised rows keep their old,
 * conservative statistics), shadows and every answer.  Queries and snapshots pinned to the old generation keep reading it,
 * so for a moment the shard is held twice: SVSB_E_NOMEM when that memory is not there, and nothing is published.  A
 * generation without tombstones keeps its buffers and only moves to the new offset. */
int svsb_compact(svsb_t* e, int64_t global_row0, uint64_t* generation);

/* _EmbeddingsMatrix.invalidate (src/svs/kb.py:861-864; call sites kb.py:984,1062,1086,1455,1523,1541). */
int svsb_invalidate(svsb_t* e);
/* Cache-hit test of get_sync / get (src/svs/kb.py:867, 880).  Returns 1 / 0. */
int svsb_is_loaded(svsb_t* e);
/* Shape of the resident matrix (embeddings_matrix.shape, used at kb.py:1191, 1629). */
int svsb_shape(svsb_t* e, int64_t* n, int32_t* d);
/* Row-norm statistics computed by the load path's norm kernel: max | ||row|| - 1 | and the number of
 * rows outside the reference's tolerance 1e-3 (src/svs/kb.py:58, src/svs/embeddings/util.py:35-38). */
int svsb_norm_stats(svsb_t* e, float* max_abs_dev, int64_t* n_out_of_tolerance);
/* Verification accessor: copy LIVE rows [row0, row0+count) of the resident matrix (and ids), in row order, back to the
 * host -- what a fresh rebuild's matrix holds at those positions. */
int svsb_read_rows(svsb_t* e, int64_t row0, int64_t count, float* rows, int64_t* emb_ids);

/* ---- the hot path: replaces superheavy() = np.dot + get_top_k + emb_id_lookup
 *      (src/svs/kb.py:1622-1627, 1184-1189; src/svs/util.py:190-203) --------------------------- */

/* q: d floats (the provider's vector as float32, NOT re-normalised, kb.py:1620).  Outputs have
 * capacity k.  *out_count = min(k, N); k <= 0 gives 0 results (util.py:198-201). */
int svsb_query(svsb_t* e, const float* q, int32_t d, int32_t k,
               float* out_scores, int64_t* out_emb_ids, int32_t* out_count);
/* The same query with several in flight from ONE host thread: submit copies q, enqueues the whole chain (query staged
 * from pinned host memory by a kernel, similarity, selection that writes the result into pinned host memory) and returns
 * at once; wait blocks for that query's result and frees the handle (every submitted handle must be waited for, also
 * after an error).  With >= 2 queries in flight the launch gaps, the serial selection and the host round trip of
 * svsb_query overlap the next query's similarity pass (src/svs/kb.py:1190: AsyncKB runs concurrent retrieves the same
 * way, one executor thread each).  At most 3 (multi-device) / SVSB_MAX_CONTEXTS (one device, default 4) can be pending;
 * a further submit blocks until one is waited for.  Multi-device engines: k <= 2048. */
typedef struct svsb_pending svsb_pending_t;
int svsb_query_submit(svsb_t* e, const float* q, int32_t d, int32_t k, svsb_pending_t** out);
int svsb_query_wait(svsb_t* e, svsb_pending_t* p, float* out_scores, int64_t* out_emb_ids, int32_t* out_count);
/* Snapshots.  The reference's retrieve keeps Python references to the (matrix, ids) pair it fetched
 * while the lock is released (src/svs/kb.py:1178-1190), so a concurrent bulk_add/bulk_del that
 * invalidates the cache (kb.py:1062, 1086) does not disturb it.  A snapshot is that pair of
 * references: it pins the generation resident at acquire time until released. */
typedef struct svsb_snapshot svsb_snap_t;
int  svsb_snapshot_acquire(svsb_t* e, svsb_snap_t** out);
void svsb_snapshot_release(svsb_snap_t* s);
int  svsb_snapshot_shape(svsb_snap_t* s, int64_t* n, int32_t* d, uint64_t* generation);
int  svsb_snapshot_rows(svsb_snap_t* s, int64_t* physical, int64_t* live);      /* as svsb_generation_rows */
int  svsb_snapshot_query(svsb_t* e, svsb_snap_t* s, const float* q, int32_t d, int32_t k,
                         float* out_scores, int64_t* out_emb_ids, int32_t* out_count);
/* Batched queries (new; the reference has no batched API -- a batch is a Python loop over retrieve,
 * src/svs/kb.py:1608-1640): Q is row-major (b, d); outputs (b, k), out_counts (b).  Same results, bit for bit, as b
 * calls of svsb_query.  Large batches on a single-device engine run as ONE dense contraction on the tensor cores
 * (fp16 coarse pass with a proven error margin, then exact fp32 re-scoring of the surviving candidates); small
 * batches, k > 1024 and multi-device engines loop over the single-query kernels. */
int svsb_query_batch(svsb_t* e, const float* Q, int32_t b, int32_t d, int32_t k,
                     float* out_scores, int64_t* out_emb_ids, int32_t* out_counts);
int svsb_snapshot_query_batch(svsb_t* e, svsb_snap_t* s, const float* Q, int32_t b, int32_t d, int32_t k,
                              float* out_scores, int64_t* out_emb_ids, int32_t* out_counts);
/* Page-locked host buffers for callers without a CUDA binding of their own.  svsb_query_batch copies straight from /
 * into caller buffers that are page-locked (these, cudaHostRegister'ed memory, torch pin_memory tensors) and stages
 * pageable ones through its own pinned buffers. */
int svsb_host_alloc(size_t bytes, void** out);
int svsb_host_free(void* p);
/* Diagnostics of the last batch chunk (<= 2048 queries): coarse candidates per query, rows re-scored exactly per
 * query, flag word per query (0 = answered by the coarse path; otherwise it took the single-query kernels). */
int svsb_batch_stats(svsb_t* e, int32_t b, int32_t* candidates, int32_t* rescored, int32_t* flags);
/* Diagnostics of the last batch chunk: query q's coarse candidate list -- up to `cap` keys (score bits in the
 * engine's order << 32 | ~row, the score being the coarse tensor-core value) -- its count (above the list's capacity,
 * SVSB_BATCH_CAND_CAP, when the list overflowed; only that many keys exist) and its eps, the bound on
 * |coarse - exact| the thresholds use.  keys and eps may be NULL. */
int svsb_batch_candidates(svsb_t* e, int32_t q, int64_t cap, uint64_t* keys, int32_t* count, float* eps);
/* Diagnostics of the last svsb_bench_run: *filter = 1 when its queries took the filter (a pass over the int8 shadow,
 * then an exact fp32 re-score of the candidate rows), 0 for the fp32 similarity kernel; *rescored = rows the last query
 * re-scored exactly (0 without the filter). */
int svsb_bench_filter_stats(svsb_t* e, int32_t* filter, int64_t* rescored);
/* The route the last svsb_bench_run's queries took: *route = 0 for the fp32 similarity kernel, 8 for the filter over the
 * int8 shadow (one scale per row; +25 % of the matrix in device memory). */
int svsb_bench_filter_route(svsb_t* e, int32_t* route);
/* How the resident generation picks the coarse pass's filter thresholds: 0 = an order statistic of a row sample that
 * bounds the true cut-off with overwhelming probability and is VERIFIED per query after the pass (default; several
 * times fewer candidates), 1 = a proven bound (the engine switches a generation to it when verification fails for
 * many queries of a batch -- rows stored in an order correlated with the queries -- or SVSB_BATCH_GUARANTEED=1).
 * Results are bit-identical in both modes.  Returns the mode, or a negative error code. */
int svsb_batch_threshold_mode(svsb_t* e);
/* Pairwise top pairs: the compute of document_top_pairwise_scores (src/svs/kb.py:1642-1671, 1208-1243) =
 * np.dot(M, M.T) + get_top_pairs (src/svs/util.py:206-233) without ever materialising the N x N scores: tensor-core
 * coarse pass over the upper triangle, one global threshold, exact fp32 re-score of the survivors.  Outputs have
 * capacity n_pairs; *out_count = min(n_pairs, N(N-1)/2).  Order: score descending, then first row ascending, then
 * second row ascending (the reference orders exact ties by descending flat index).  Multi-device engines split the
 * pairs over the devices (each runs the triangle of its own shard and rectangles against blocks of its peers' rows, with
 * its own threshold) and merge the per-device lists on device 0: the result equals the single-device engine's bit for
 * bit.  SVSB_E_INVALID: tombstoned rows, rows far from unit norm, n_pairs above 2^22; SVSB_E_NOMEM: more near-tied pairs
 * than the candidate lists hold -- refusals the reference's host path still answers. */
int svsb_top_pairs(svsb_t* e, int64_t n_pairs, float* out_scores, int64_t* out_emb_ids_a, int64_t* out_emb_ids_b,
                   int64_t* out_count);
int svsb_snapshot_top_pairs(svsb_t* e, svsb_snap_t* s, int64_t n_pairs, float* out_scores, int64_t* out_emb_ids_a,
                            int64_t* out_emb_ids_b, int64_t* out_count);
/* Selection only: get_top_k (src/svs/util.py:190-203) on a host score vector, run by the same
 * selection kernels.  out_index receives row indices. */
int svsb_topk_scores(svsb_t* e, const float* scores, int64_t n, int32_t k,
                     float* out_scores, int64_t* out_index, int32_t* out_count);

/* ---- measurement support (device-resident inputs; used by bench.py and the parity tests) ------ */

/* Upload nq query vectors (row-major (nq, d)) to every device once. */
int svsb_bench_set_queries(svsb_t* e, const float* Q, int32_t nq, int32_t d);
/* Run `iters` single-query retrieves back to back, cycling through the uploaded queries, everything
 * device-resident, timed with CUDA events on the launching stream(s).  Returns total milliseconds
 * (max over devices), the number of kernel launches issued and, when gemv_ms != NULL, the duration of the
 * similarity-kernel launches on device 0: one launch in 8 is bracketed by its own pair of events inside the same
 * timed loop and *gemv_ms = (mean bracketed launch) x iters (the roofline numerator's denominator). */
int svsb_bench_run(svsb_t* e, int32_t k, int32_t iters, float* total_ms, float* gemv_ms, int64_t* launches);
/* Same through the batched path: per iteration ONE batch of all uploaded queries (<= 2048), device-resident.
 * coarse_ms (optional): summed duration of the tensor-core filter pass, bracketed by its own events. */
int svsb_bench_run_batch(svsb_t* e, int32_t k, int32_t iters, float* total_ms, float* coarse_ms, int64_t* launches);
/* Result of query qi of the last svsb_bench_run_batch iteration (checks that the timed path computes the answer). */
int svsb_bench_batch_result(svsb_t* e, int32_t qi, int32_t k, float* out_scores, int64_t* out_emb_ids, int32_t* out_count,
                            int32_t* out_flag);
/* Development aid: %globaltimer phase stamps (ns) of one selection-kernel run with uploaded query qi. */
int svsb_debug_select_phases(svsb_t* e, int32_t qi, int32_t k, uint64_t* stamps16);
/* Result of the last bench query (for checking that the timed path computes the right thing). */
int svsb_bench_last_result(svsb_t* e, int32_t k, float* out_scores, int64_t* out_emb_ids, int32_t* out_count);

/* ---- sharded deployment: one process per GPU (SURVEY.md section 8e) -----------------------------
 * Each process owns ONE device and the rows [global_row0, global_row0 + n) of the matrix, in scan order.
 * Two ways to do the one exchange step.  (1) Collective: the library does the compute on the caller's stream and
 * the caller (torch.distributed / NCCL) all-gathers one packed record per query per rank, then
 * svsb_enqueue_merge_records (k > 2048: svsb_enqueue_merge_sorted_records).  (2) Fused ("peer exchange", below): the kernels themselves move the records over
 * NVLink peer memory; the caller only exchanges 64-byte IPC handles once.  None of the svsb_enqueue_* / svsb_xchg_* /
 * svsb_*_peer entry points is re-entrant: one host thread drives a shard engine.
 * Record layout: 2*k+1 int64 words = [ keys (k, uint64: ordered score << 32 | ~global_row) |
 *                                      embeddings.id (k) | count (int32 in the low half of the last word) ]. */
int svsb_set_shard(svsb_t* e, int64_t global_row0);           /* call before svsb_load_*          */
/* flags: bit 0 = bracket the similarity kernel with timing events (svsb_kernel_time_collect); bit 1 = pipelined:
 * the similarity kernel runs on `stream` leaving one SM free and the one-CTA selection kernel runs on an engine-owned
 * side stream, so the selection of query i overlaps the similarity pass of query i+1 when consecutive calls
 * alternate `slot`.  With bit 1 the record is complete only after svsb_enqueue_join(e, stream).
 * Any k >= 1; the record has room for k entries and holds min(k, rows of this shard), sorted descending.  k > 2048
 * (full rankings) sorts all of the shard's keys after the similarity pass; it always runs unpipelined on `stream`
 * (bit 1 is ignored) and needs sort scratch of next_pow2(rows) keys in the slot's workspace (SVSB_E_NOMEM if that
 * cannot be allocated; nothing is enqueued then).  Merge such records with svsb_enqueue_merge_sorted_records. */
int svsb_enqueue_local_topk(svsb_t* e, void* stream, int32_t slot, const float* d_query, int32_t k,
                            int64_t* d_record, int32_t flags);
/* Batched form: local top-k records of b device-resident queries d_Q[b][ld] (ld = d rounded up to 4, zero padded)
 * on `stream`.  Large batches take the tensor-core coarse pass + exact refine (same bits as the single-query kernels),
 * flagged queries / small batches / k > 1024 take the single-query kernels.  *n_fallback = queries that did.
 * Synchronises `stream` once per 2048 queries. */
int svsb_batch_local_records(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, int64_t* d_records,
                             int32_t* n_fallback);
/* Batches with ONE filter threshold per query for all ranks (the sharded form of retrieve_many; reference: a loop of
 * superheavy(), src/svs/kb.py:1622-1627, over a matrix that no longer lives in one place).  With svsb_batch_local_records
 * every rank finds its OWN top k, so the per-batch costs do not shrink with the shard; here each rank only keeps and
 * re-scores what can reach the GLOBAL top k.  Per batch of b <= 2048 queries, on every rank, nothing synchronises:
 *   1. svsb_batch_sample_tops      -> d_tops[b][32]: the 32 largest coarse scores of this rank's sample, descending
 *   2. the caller all-gathers them -> d_tops_all[world][b][32]
 *   3. svsb_batch_global_records   -> threshold = (sample_rank-th largest of the union) - 2 eps, filter pass, exact
 *      re-score of every candidate, records [keys(rec_cap) | ids(rec_cap) | count, ver], 2*rec_cap+1 words (count may be
 *      < k; count -1 = this rank could not answer the query; ver = candidates provably above the threshold's margin).
 *      rec_cap <= k entries are shipped per rank -- a shard holds ~k/world of the global top k, so records an eighth
 *      the size do on 8 GPUs; a rank with more sets bit 30 of count and the merge accepts the query only if that
 *      list's last shipped entry does not make the global top k (then nothing behind it can).
 *   4. the caller all-gathers the records; svsb_enqueue_merge_batch_records(verify_k = min(k, global rows)) merges
 *      and VERIFIES: out_count -1 (on every rank alike) = redo this query with the exact path (svsb_query_peer /
 *      svsb_enqueue_local_topk); otherwise the result equals the single-query kernels' bit for bit.
 * svsb_batch_global_probe tells whether this rank can take part (eligible) and what the caller needs to choose ONE
 * sample_rank and ONE max_row_norm for all ranks: with f = max over ranks of sample_rows / local_rows and
 * lambda = min(k, global rows) * f, sample_rank = ceil(lambda + 6 sqrt(lambda) + 4) must be <= 32 (else use
 * svsb_batch_local_records); max_row_norm = the largest over the ranks.  Steps 1 and 3 of one batch must not be
 * interleaved with another batch on the same engine. */
int svsb_batch_global_probe(svsb_t* e, int32_t k, int32_t* eligible, int64_t* sample_rows, int64_t* local_rows, float* max_row_norm);
int svsb_batch_sample_tops(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, float max_row_norm, float* d_tops);
int svsb_batch_global_records(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, const float* d_tops_all,
                              int32_t world, int32_t sample_rank, int32_t rec_cap, int64_t* d_records);
/* The same batch protocol with BOTH exchanges fused into the kernels over NVLink / NVSwitch peer memory: no collective
 * call.  Every rank owns a BATCH WINDOW (svsb_bxchg_create; 64-byte CUDA IPC handle, exchanged once and opened with
 * svsb_bxchg_connect; svsb_bxchg_connect_local for several shard engines inside one process); the kernel that extracts a
 * rank's sample maxima stores them into every rank's window, the kernel that sorts a rank's exact candidates does the
 * same with its records; each ends with a system-scope release of the batch's sequence number, and the consumers (union
 * threshold, verifying merge) run behind a one-CTA kernel that acquires the flags of its own window.
 * svsb_batch_peer enqueues one whole batch (b <= 2048) on `stream`: device queries in, device (b, k) results out,
 * out_counts[q] = k', -1 (redo this query with the exact path, as svsb_enqueue_merge_batch_records) or -2 (a peer's part
 * did not arrive within SVSB_XCHG_TIMEOUT_MS).  Every rank calls it with the same arguments in the same order.
 * rec_cap (<= the window's) / sample_rank / max_row_norm as in svsb_batch_global_records.  svsb_batch_peer_prepare sizes
 * the workspace up front (needed only when several shard engines share one process). */
int svsb_bxchg_create(svsb_t* e, int32_t world, int32_t rank, int32_t rec_cap, void* handle_out);
int svsb_bxchg_connect(svsb_t* e, const void* handles);
int svsb_bxchg_connect_local(svsb_t* e, svsb_t* const* engines);
int svsb_bxchg_disconnect(svsb_t* e);
int svsb_batch_peer_prepare(svsb_t* e, int32_t b, int32_t k);
int svsb_batch_peer(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, float max_row_norm, int32_t sample_rank,
                    int32_t rec_cap, float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_counts, int32_t flags);
/* flags bit 0 = pipelined: the batch's verifying merge (the only step that waits for the peers' records) is enqueued
 * behind the FIRST phase of the next svsb_batch_peer call on this engine, or by svsb_batch_peer_flush -- the peers get
 * that long to deliver, which hides the ranks' skew in a stream of batches.  The outputs are complete after whichever
 * enqueues the merge. */
int svsb_batch_peer_flush(svsb_t* e, void* stream);
/* ---- peer exchange: the exchange step fused into the kernels, over NVLink / NVSwitch peer memory ----------
 * Replaces "all-gather the records over NCCL, then merge" for single queries: every rank owns a GATHER WINDOW in its
 * HBM (slots x world records + one flag word per record); the selection kernel's epilogue stores its record into the
 * window of EVERY rank with plain peer stores and publishes it with a system-scope release store of the query's
 * sequence number; the merge kernel of each rank acquires the `world` flags of its own window and merges.  No
 * collective library call and no extra launch sit between a shard's local top-k and the global answer.
 * SPMD contract: all ranks issue the same sequence of svsb_enqueue_query_peer / svsb_query_peer calls (the sequence
 * number is implicit), each rank in stream order.
 *   svsb_xchg_create        allocates this rank's window (k <= k_max <= 2048, world <= 16) and returns its CUDA IPC
 *                           handle (64 bytes) for the launcher to all-gather (torch.distributed, any backend);
 *   svsb_xchg_connect       opens the peers' windows: handles = world x 64 bytes, rank order (own entry ignored);
 *   svsb_xchg_connect_local same for engines living in THIS process (tests; one process driving several GPUs). */
int svsb_xchg_create(svsb_t* e, int32_t world, int32_t rank, int32_t k_max, void* ipc_handle_out);
int svsb_xchg_connect(svsb_t* e, const void* ipc_handles);
int svsb_xchg_connect_local(svsb_t* e, svsb_t* const* engines);
/* Orderly shutdown: every rank disconnects (waits for its own queries, unmaps the peers' windows), the launcher
 * barriers, then the engines are destroyed -- no rank frees a window another rank still has mapped. */
int svsb_xchg_disconnect(svsb_t* e);
/* One query, device resident: similarity on `stream`, selection + push + waiting merge on `stream` (flags bit 1 clear)
 * or on the engine's side stream with one SM reserved for them (bit 1 set: overlaps the next query's similarity
 * pass; outputs are complete after svsb_enqueue_join).  Bit 0: time the similarity kernel (svsb_kernel_time_collect).
 * Outputs (device or pinned host pointers): GLOBAL top-k, identical on every rank; *d_out_count = min(k, N). */
int svsb_enqueue_query_peer(svsb_t* e, void* stream, const float* d_query, int32_t k,
                            float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_count, int32_t flags);
/* One query, host buffers in and out, synchronous (the sharded counterpart of svsb_query; replaces a6 + a7 of
 * SURVEY.md section 8 on a row-sharded matrix): a staging kernel reads the query from pinned host memory, similarity,
 * selection + push, waiting merge that writes the result straight into pinned host memory, one stream synchronize.
 * SVSB_E_STATE if a peer's record does not arrive within SVSB_XCHG_TIMEOUT_MS (default 30 000): the sequence is then
 * broken and the exchange must be re-created on every rank. */
int svsb_query_peer(svsb_t* e, const float* q, int32_t d, int32_t k,
                    float* out_scores, int64_t* out_emb_ids, int32_t* out_count);
/* The same with up to 3 queries in flight from the host thread that drives the shard engine (SPMD: every rank issues
 * the same sequence of submits; waits are local, oldest first).  Query j+1's similarity pass overlaps query j's selection,
 * exchange, merge and host round trip: selection + push and the waiting merge run on the engine's side stream with one
 * SM reserved for them.  Do not interleave with svsb_enqueue_query_peer while tickets are pending. */
int svsb_query_peer_submit(svsb_t* e, const float* q, int32_t d, int32_t k, int32_t* ticket);
int svsb_query_peer_wait(svsb_t* e, int32_t ticket, float* out_scores, int64_t* out_emb_ids, int32_t* out_count);
/* Development aid: with SVSB_XCHG_STAMPS=1 in the environment at svsb_xchg_create, the selection and merge kernels of
 * the synchronous svsb_query_peer stamp %globaltimer (ns) into a ring of 1024 queries x 40 words: per query
 * [16 selection stamps as svsb_debug_select_phases | seq, merge start, merge done, -, time rank r's flag was seen x world]. */
int svsb_xchg_read_stamps(svsb_t* e, uint64_t* out, int64_t capacity_words);
/* Make `stream` wait for everything the pipelined svsb_enqueue_local_topk / svsb_enqueue_query_peer calls have issued
 * on the side stream (it also enqueues the last peer query's deferred merge). */
int svsb_enqueue_join(svsb_t* e, void* stream);
/* d_records: all-gathered records, [n_lists][batch][2k+1].  Outputs [batch][k], [batch][k], [batch]. */
int svsb_enqueue_merge_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t batch,
                               int32_t k, float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_counts);
/* The same for the records of svsb_batch_global_records: a query comes out with count -1 when any rank's record says
 * -1 or the ranks' verification counts add up to less than verify_k. */
int svsb_enqueue_merge_batch_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t batch,
                                     int32_t rec_cap, int32_t k, int32_t verify_k, float* d_out_scores, int64_t* d_out_ids,
                                     int32_t* d_out_counts);
/* Any k: merge `n_lists` records of `cap` entries each, [n_lists][2*cap+1] words, every one sorted descending (what
 * svsb_enqueue_local_topk writes; keys carry the global row, so keys are unique across ranks and ties break by ascending
 * row).  Outputs: the top min(k, sum of counts) entries in d_out_scores[k] / d_out_ids[k] and that number in
 * *d_out_count.  Each rank's record must hold everything of its shard that can reach the top k: cap >= min(k, rows of
 * the largest shard).  A record whose count is negative or above cap (e.g. RECORD_TRUNCATED, bit 30, of the batch
 * records) cannot be merged exactly: *d_out_count = -1 and nothing else is written.  Nothing is verified beyond that. */
int svsb_enqueue_merge_sorted_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t cap, int32_t k,
                                      float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_count);
/* ---- pairwise top pairs over the ranks' shards (the sharded form of svsb_top_pairs) --------------------------------
 * The result equals svsb_top_pairs of one single-device engine over the global matrix bit for bit: scores, ids, order.
 * Rank r runs its share of a static plan over the world's shards (the triangle of its own shard, rectangles against
 * 1024-row blocks of its peers' fp16 rows, copied over CUDA IPC) with its own threshold, re-scores its survivors
 * exactly (the peer's row read over the mapping) and keeps its top list; the caller all-gathers the lists and every rank
 * merges them.  No kernel waits on a flag: a missing peer blocks the caller's collective, never the GPU.  Per call, on
 * every rank, in this order:
 *   svsb_pairs_export        pins the resident generation of this single-device engine, builds its fp16 shadow and
 *                            writes a descriptor of SVSB_PAIRS_DESC_BYTES (CUDA IPC handles of the fp32 rows, the fp16
 *                            shadow and the ids; n, d, global first row; an empty shard has no handles) for the caller to
 *                            all-gather.  *max_dev_out = max | ||row|| - 1 | of the shard, *rows_out = its rows.  Refuses
 *                            as svsb_top_pairs: SVSB_E_NOT_LOADED, tombstoned rows (SVSB_E_INVALID); and an engine over
 *                            several devices (SVSB_E_INVALID).  Only when disconnected (SVSB_E_STATE otherwise); drops
 *                            the previously pinned generation.
 *   svsb_pairs_connect       opens the peers' descriptors (world x SVSB_PAIRS_DESC_BYTES in rank order, own entry
 *                            ignored; world <= 16); svsb_pairs_connect_local takes the engines of ranks living in THIS
 *                            process instead (each exported).  Both check that d agrees and that the ranks' rows are
 *                            contiguous in rank order.  Rows of the protocol are global, counted from rank 0's first.
 *   (once per load: export, all-gather, connect, barrier; then any number of the calls below)
 *   svsb_pairs_local         this rank's list: min(n, survivors) pairs in the final order (score desc, first row asc,
 *                            second row asc), rows in d_rows_a < d_rows_b, into device buffers of capacity n, where n =
 *                            min(n_pairs, N(N-1)/2) of the GLOBAL N; *out_count (host) = entries.  max_row_norm must be
 *                            the same on every rank: the max over ranks of 1 + max_dev.  Runs behind the work already on
 *                            `stream` and returns when its outputs are complete.  SVSB_E_INVALID: rows far from unit norm,
 *                            n above 2^22; SVSB_E_NOMEM: more near-tied pairs than the candidate lists hold (a rank may
 *                            refuse alone: the caller must agree on the outcome before the exchange).
 *   (the caller all-gathers the counts and the lists, padded to stride = max count: list l at [l * stride ..))
 *   svsb_pairs_merge         merges the world lists on `stream` into the top n, rows mapped to embeddings.id; *d_out_count
 *                            (device) = n.
 * Teardown (and before re-exporting after a reload): every rank's last pairs call has returned, every rank calls
 * svsb_pairs_disconnect (unmaps the peers' shards, releases the pinned generation), the launcher barriers, and only then
 * are engines destroyed -- no rank frees a shard another rank can still read. */
#define SVSB_PAIRS_DESC_BYTES 256
int svsb_pairs_export(svsb_t* e, float* max_dev_out, int64_t* rows_out, void* desc_out);
int svsb_pairs_connect(svsb_t* e, int32_t world, int32_t rank, const void* descs);
int svsb_pairs_connect_local(svsb_t* e, int32_t world, int32_t rank, svsb_t* const* engines);
int svsb_pairs_local(svsb_t* e, void* stream, int64_t n_pairs, float max_row_norm, float* d_scores, int64_t* d_rows_a,
                     int64_t* d_rows_b, int64_t* out_count);
int svsb_pairs_merge(svsb_t* e, void* stream, const float* d_scores, const int64_t* d_rows_a, const int64_t* d_rows_b,
                     const int32_t* d_counts, int32_t world, int64_t stride, int64_t n, float* d_out_scores,
                     int64_t* d_out_ids_a, int64_t* d_out_ids_b, int32_t* d_out_count);
int svsb_pairs_disconnect(svsb_t* e);
/* Sum (ms) of the similarity-kernel durations bracketed by svsb_enqueue_local_topk(time_kernel=1) since the
 * last collect; waits for them to finish. */
int svsb_kernel_time_collect(svsb_t* e, float* ms);

/* ---- stateless launchers on raw device pointers (one process per GPU; pointers may come from
 *      torch tensors' data_ptr(), stream from torch.cuda.current_stream().cuda_stream) ---------- */

typedef struct svsb_workspace svsb_ws_t;
int  svsb_ws_create(int device, int64_t n_rows, int32_t k_max, svsb_ws_t** out);
void svsb_ws_destroy(svsb_ws_t* ws);
/* Local top-k of one shard: keys (64-bit, order-preserving score in the high word, ~global_row in the
 * low word) and embeddings.ids of the min(k, n) best rows, sorted.  All pointers are device pointers. */
int svsb_launch_local_topk(svsb_ws_t* ws, void* stream, const float* d_matrix, int64_t n, int32_t d,
                           int32_t ld, const int64_t* d_emb_ids, int64_t global_row0, const float* d_query,
                           int32_t k, uint64_t* d_out_keys, int64_t* d_out_ids, int32_t* d_out_count);
/* Merge G gathered candidate lists (each `stride` entries long, counts[g] valid) into the global
 * top-k: scores, ids.  Used after the NCCL all-gather of the per-rank lists. */
int svsb_launch_merge(svsb_ws_t* ws, void* stream, const uint64_t* d_keys, const int64_t* d_ids,
                      const int32_t* d_counts, int32_t n_lists, int32_t stride, int32_t k,
                      float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_count);

const char* svsb_last_error(void);
const char* svsb_version(void);
/* Number of kernel launches this process has issued through the library (for bench.py's gpu_launches). */
int64_t svsb_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SVSB200_H */
