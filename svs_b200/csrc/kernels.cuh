// Internal C++ interface between the engine (engine.cu) and the kernels.
#pragma once
#include "common.cuh"

namespace svsb {

// Launch counter (svsb_launch_count): every kernel launch of the library goes through count_launch().
void count_launch(int n = 1);

// Programmatic dependent launch for the one-query-in-flight chains (stage query -> similarity -> selection -> merge):
// while set (per host thread), the launchers below mark their kernel "programmatic stream serialization allowed", so
// it may start while the previous kernel of the stream is still running; the kernels call pdl_wait() before they
// touch anything the previous kernel produces and pdl_trigger() as early as their successor may be scheduled.
// Without the attribute both are no-ops, so every other path is unchanged.
void set_pdl(bool on);
bool pdl_enabled();
struct PdlScope { bool prev; explicit PdlScope(bool on) : prev(pdl_enabled()) { set_pdl(on); } ~PdlScope() { set_pdl(prev); } };

#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    if (pdl_enabled()) {
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#endif

// ---- K1: similarity (fp32 GEMV) -------------------------------------------------------------
// scores[r] = dot(M[r, :], q) for r < n, and gmax[r >> group_shift] = max(key(score, r)) via atomics.
// M is row-major with leading dimension ld floats (ld % 4 == 0, rows 16-byte aligned, padding zero);
// q has ld floats (padding zero).  gmax must be zero on entry.
// variant: 0 = auto, 1 = LDG.128 streaming kernel, 2 = TMA-bulk (cp.async.bulk + mbarrier ring) kernel.
// tune_a/tune_b: variant-specific knobs (0 = default), see gemv.cu.  reserve_sms: SMs the persistent grid leaves
// free (the pipelined paths run the previous query's selection kernel there, concurrently).
// live (optional): one byte per row, 0 = tombstoned (svsb_apply_mutations): such a row's score is written as
// dead_score(), whose key sorts below every real score's, so it is selected only after all live rows.
cudaError_t launch_gemv(cudaStream_t st, int device, const float* M, int64_t n, int d, int ld,
                        const float* q, float* scores, u64* gmax, int group_shift,
                        int variant = 0, int tune_a = 0, int tune_b = 0, int reserve_sms = 0,
                        const uint8_t* live = nullptr);

// K1f, the fp16 filter (gemv.cu, DESIGN.md section 4): launch_filter writes launch_gemv's outputs as COARSE values from
// the shadow M16[n][ld16] = fp16(M * 2^12) (launch_rows_to_f16) and the fp32 query q[ld]; launch_filter_refine then
// (1 CTA) sets the candidate threshold state[0] from the group maxima and the bound
// eps = eps_coef * ||q|| * max_row_norm + 1e-8 on |coarse - exact|, and (many CTAs) re-scores every candidate exactly --
// the bits launch_gemv writes -- leaving scores / gmax such that launch_select returns launch_gemv's top-kk.
// state: 2 device words, state[1] = rows re-scored.  ld <= FILTER_MAX_LD.
constexpr int FILTER_MAX_LD = 3072;
cudaError_t launch_filter(cudaStream_t st, int device, const void* M16, int64_t n, int ld, int ld16, const float* q,
                          float* scores, u64* gmax, int group_shift, int reserve_sms = 0, const uint8_t* live = nullptr);
// e8: null for the fp16 filter; the int8 shadow's error word E for launch_filter8's coarse scores (then the threshold
// uses the int8 bound, gemv.cu filter_threshold_kernel).
cudaError_t launch_filter_refine(cudaStream_t st, int device, const float* M, int64_t n, int ld, const float* q, float* scores,
                                 u64* gmax, int group_shift, int kk, float eps_coef, float max_row_norm, const float* e8,
                                 const uint8_t* live, uint32_t* state);
// K1f8, the int8 filter (gemv.cu, DESIGN.md section 4): launch_filter's contract over the int8 shadow M8[n][ld8] with
// one scale per row (launch_rows_to_i8).  ld8 % 16 == 0, ld <= FILTER_MAX_LD.
cudaError_t launch_filter8(cudaStream_t st, int device, const void* M8, const float* scale8, int64_t n, int ld, int ld8,
                           const float* q, float* scores, u64* gmax, int group_shift, int reserve_sms = 0,
                           const uint8_t* live = nullptr);
// M8[r] = round(M[r] / scale8[r]) with scale8[r] = max|M[r][.]| / 127, zero padded; *emax (a float, only raised) >= every
// converted row's ||M[r] - scale8[r] * M8[r]||.  ld % 4 == 0, ld8 % 16 == 0, ld8 >= ld.
cudaError_t launch_rows_to_i8(cudaStream_t st, int device, const float* M, int64_t n, int ld, void* M8, int ld8, float* scale8,
                              float* emax);
// the bound's coefficient for d components (fp16 operands, fp32 accumulation; DESIGN.md section 6, step 4)
inline float coarse_eps_coef(int d) {
    return 9.765625e-4f + 2.384185791015625e-7f + (float)d * (2.384185791015625e-7f + 1.1920928955078125e-7f);
}

// b queries Q[b][ld] in ONE pass over the matrix: scores[q * n_stride + r], gmax[q * g_stride + (r >> shift)] (zero on
// entry), bit-identical to b launch_gemv calls.  cudaErrorInvalidConfiguration: rows too long (ld > 3072) or b larger
// than 8 warps' worth of queries (8 * gemv_mq_queries_per_warp(ld)); the caller chunks / falls back.
int gemv_mq_queries_per_warp(int ld);
cudaError_t launch_gemv_mq(cudaStream_t st, int device, const float* M, int64_t n, int d, int ld, const float* Q, int b,
                           float* scores, int64_t n_stride, u64* gmax, int64_t g_stride, int group_shift,
                           const uint8_t* live = nullptr, int reserve_sms = 0);

// ---- K3/K4: exact top-k ---------------------------------------------------------------------
// Inputs: scores[n], gmax[ceil(n >> shift)] (consumed and reset to zero), ids[n] (may be null: ids = rows).
// Outputs (device): out_keys[k] (key with GLOBAL row = row0 + local row), out_scores[k], out_ids[k],
// *out_count = min(k, n).  cand is scratch of cand_cap entries, cand_cap >= min(n, K_FAST_MAX << shift) + K_FAST_MAX.
// Requires 1 <= k <= K_FAST_MAX.
// push (optional): the fused exchange step of the one-process-per-GPU deployment -- the epilogue also stores the
// record (keys, ids, count) into every rank's gather window over peer memory (NVLink / NVSwitch P2P stores) and then
// publishes it there with a system-scope release store of the query's sequence number (see PeerPush).
struct PeerPush;
cudaError_t launch_select(cudaStream_t st, const float* scores, int64_t n, u64* gmax, int group_shift,
                          int k, const int64_t* ids, int64_t row0, u64* cand, int64_t cand_cap,
                          u64* out_keys, float* out_scores, int64_t* out_ids, int32_t* out_count,
                          u64* dbg = nullptr,    // dbg: optional 16 x u64 of %globaltimer phase stamps
                          const PeerPush* push = nullptr);
// The same for b queries in one launch (one CTA per query, on b different SMs): query q reads scores + q * s.scores,
// gmax + q * s.gmax, uses cand + q * s.cand and writes out_keys + q * s.keys, out_scores + q * s.oscores,
// out_ids + q * s.ids, out_count + q * s.count (strides in elements of the respective array).
struct SelectStrides { int64_t scores = 0, gmax = 0, cand = 0, keys = 0, oscores = 0, ids = 0, count = 0; };
cudaError_t launch_select_batch(cudaStream_t st, int b, const SelectStrides& s, const float* scores, int64_t n, u64* gmax, int group_shift,
                                int k, const int64_t* ids, int64_t row0, u64* cand, int64_t cand_cap,
                                u64* out_keys, float* out_scores, int64_t* out_ids, int32_t* out_count);

// Large-k path (k > K_FAST_MAX): sort all n keys.  sortbuf has next_pow2(n) entries.  Also zeroes gmax.
cudaError_t launch_fullsort_topk(cudaStream_t st, const float* scores, int64_t n, u64* gmax, int group_shift,
                                 int64_t k, const int64_t* ids, int64_t row0, u64* sortbuf,
                                 u64* out_keys, float* out_scores, int64_t* out_ids, int32_t* out_count);

// gmax from a score vector alone (svsb_topk_scores: selection without the GEMV).
cudaError_t launch_groupmax(cudaStream_t st, int device, const float* scores, int64_t n, u64* gmax, int group_shift);

constexpr int MERGE_WINDOW_TIMED_OUT = -2;          // out_count of a merge whose peers' records did not arrive
// Merge n_lists candidate lists (keys carry global rows; ids are the payload) into the top-k.
// scratch: u64[next_pow2(n_lists * stride)] + int64[same] when n_lists * stride > K_FAST_MAX (else unused).
cudaError_t launch_merge(cudaStream_t st, const u64* keys, const int64_t* ids, const int32_t* counts,
                         int n_lists, int stride, int k, u64* scratch_keys, int64_t* scratch_ids,
                         float* out_scores, int64_t* out_ids, int32_t* out_count);

// Strided / batched form (one CTA per query of the batch); strides in elements.  scratch (big case only):
// batch * n_lists * cap entries each.
cudaError_t launch_merge_ex(cudaStream_t st, const u64* keys, const int64_t* ids, const int32_t* counts,
                            int n_lists, int cap, int k, int batch, int64_t list_stride, int64_t batch_stride,
                            int64_t count_list_stride, int64_t count_batch_stride,
                            u64* scratch_keys, int64_t* scratch_ids,
                            float* out_scores, int64_t* out_ids, int32_t* out_count,
                            int verify_k = -1,    // >= 0: count words are [count, ver] pairs, see MergeLayout (select.cu)
                            const int* abort_flag = nullptr);   // device word; non-zero: every out_count = MERGE_WINDOW_TIMED_OUT

// Any k: merge n_lists lists, each SORTED descending with unique keys.  List l holds counts[l * count_stride] <= cap
// entries at keys / ids [l * list_stride ..) (strides in elements of the respective array).  out_count = min(k, sum of
// counts), or -1 when a count is negative or above cap (a truncated list: the answer is unknown, nothing is written).
cudaError_t launch_merge_sorted_big(cudaStream_t st, const u64* keys, const int64_t* ids, const int32_t* counts, int n_lists,
                                    int64_t cap, int64_t list_stride, int64_t count_stride, int64_t k, float* out_scores,
                                    int64_t* out_ids, int32_t* out_count);

// ---- peer exchange (select.cu): candidate records pushed into every rank's window, merged after a flag wait ----
// A window holds `slots` x `world` records of rec_words = 2*cap + 2 u64 words: [keys(cap) | ids(cap) | count | pad],
// plus slots x world u64 flags.  Query number seq (1, 2, ...) uses slot seq % slots; flag (slot, r) == seq means
// rank r's record for that query is complete in THIS window.
constexpr int XCHG_MAX_RANKS = 16;
struct PeerPush {
    int world = 0, cap = 0;
    unsigned long long seq = 0;
    u64* rec[XCHG_MAX_RANKS];       // rec[p]: where THIS rank's record goes in rank p's window (slot already applied)
    u64* flag[XCHG_MAX_RANKS];      // flag[p]: rank p's flag word for (slot, this rank)
};
// Load every kernel of the peer paths onto the current device now (lazy module loading would otherwise synchronise
// the context at a kernel's first launch -- while a merge kernel of the same process may be spinning on a flag).
cudaError_t preload_gemv_kernels();
cudaError_t preload_peer_kernels();
cudaError_t preload_batch_kernels();     // batch.cu
cudaError_t preload_coarse_kernels();    // coarse.cu
cudaError_t preload_merge_kernels();     // select.cu
// d_q[0..ld) = host_q_mapped[0..ld) (pinned host memory, read by a kernel: no copy-engine operation).  ld % 4 == 0.
cudaError_t launch_stage_query(cudaStream_t st, const float* host_q_mapped, float* d_q, int ld);
// Record with count 0 (this rank owns no rows): same publication protocol, one small CTA.
cudaError_t launch_push_empty(cudaStream_t st, const PeerPush& push);
// One CTA: wait until flags[0..world) >= seq (ld.acquire.sys), then merge the world lists of the window slot
// (coherent loads: the data was written by remote GPUs) into the top-k.  scratch as launch_merge (world*cap > 2048).
// A flag that does not arrive within timeout_ns (a peer died or left the SPMD call sequence) ends the kernel with
// *out_count = MERGE_WINDOW_TIMED_OUT instead of hanging the GPU.
cudaError_t launch_merge_window(cudaStream_t st, const u64* slot_base, const u64* flags, unsigned long long seq,
                                int world, int cap, int k, unsigned long long timeout_ns, u64* scratch_keys, int64_t* scratch_ids,
                                float* out_scores, int64_t* out_ids, int32_t* out_count,
                                u64* stamps = nullptr);   // optional 24 x u64: [seq, t_start, t_done, -, t_flag_seen[world]] (%globaltimer ns)

// ---- K0: load path ---------------------------------------------------------------------------
// Row L2 norms; optionally divide rows by their norm.  stats[0] = float bits of max | ||row|| - 1 |
// (atomicMax on non-negative floats), stats[1] = number of rows with deviation > tol.  stats must be zeroed.
cudaError_t launch_row_norms(cudaStream_t st, int device, float* M, int64_t n, int d, int ld, int normalize,
                             float tol, float* norms_or_null, u64* stats);
// Counter-based synthetic rows (oracle/svs_oracle.py counter_uniform_rows) + ids.
cudaError_t launch_synth(cudaStream_t st, int device, float* M, int64_t n, int d, int ld, uint64_t seed,
                         int64_t global_row0, int64_t* ids, int64_t id0, int64_t id_step);

// ---- K2: batched queries = coarse tensor-core contraction + exact refine (coarse.cu, batch.cu) -----------
constexpr int COARSE_MAX_BATCH = 2048;              // queries per coarse launch (thresholds live in shared memory)
constexpr int COARSE_TILE_ROWS = 128;               // rows per coarse tile (UMMA M)
constexpr int COARSE_TILE_QUERIES = 256;            // queries per coarse tile (UMMA N); batches are padded to it
constexpr float COARSE_OPERAND_SCALE = 4096.0f;     // 2^12 on both operands: keeps fp16 components normal, exact to undo
constexpr int COARSE_DEFAULT_CTAS = 1;               // 1 = single-CTA tiles, 2 = CTA pairs (cta_group::2); env SVSB_COARSE_CTAS
constexpr int REFINE_SURVIVOR_CAP = 4096;           // exact re-scores per query the refine kernel can hold

// M16[r][0..ld16) = fp16(M[r][.] * 2^12), zero padded.  ld % 4 == 0, ld16 % 8 == 0, ld16 >= ld.
cudaError_t launch_rows_to_f16(cudaStream_t st, int device, const float* M, int64_t n, int ld, void* M16, int ld16);
// Q16 (b_pad rows, rows >= b zero) from fp32 queries Q[b][ldq]; eps[q] = eps_coef * ||q|| * max_row_norm + 1e-8,
// thr[q] = +inf, flags[q] = 1 for queries the coarse path must not handle (non-finite / huge norm).
cudaError_t launch_queries_to_f16(cudaStream_t st, const float* Q, int b, int b_pad, int d, int ldq, void* Q16, int ld16,
                                  float eps_coef, float max_row_norm, float* eps, float* thr, int32_t* flags,
                                  int32_t* cand_cnt = nullptr);   // optional: cand_cnt[0..b_pad) = 0
// mode 0: filter -- every (row, query) whose coarse score >= thr[query] is appended to cand[query][..cand_cap)
//         (key = ordered coarse score << 32 | ~row), cand_cnt[query] counts ALL survivors (may exceed cand_cap).
// mode 1: sample -- coarse scores of row tiles 0, tile_stride, 2*tile_stride, ... (n_tiles of them), rounded DOWN to
//         fp16, go to sample[query][sample_rows] (__half); rows beyond n read as -inf.
// q_rows > 0: Q16 holds only q_rows (<= b_pad) rows, the rest of the padded batch reads as zero.
// tri_q0 >= 0: pairwise mode -- Q16 is the matrix itself from row tri_q0 on; only pairs (query row < matrix row)
// count, tiles on or below the diagonal are skipped.
cudaError_t launch_coarse_gemm(cudaStream_t st, int device, int mode, const void* M16, int64_t n, const void* Q16, int b_pad,
                               int ld16, int n_tiles, int tile_stride, const float* thr, u64* cand, int32_t* cand_cnt,
                               int cand_cap, void* sample, int64_t sample_rows, int64_t q_rows = 0, int64_t tri_q0 = -1);
// thr[q] = (rank-th largest of sample[q][0..sample_rows)) - 2 eps[q] for q < b (one CTA per query).
// sample: fp16 (coarse scores rounded down), as the coarse kernel's mode 1 writes it.
// rank == kk: a guaranteed lower bound of (kk-th largest coarse score of all rows) - 2 eps.  rank < kk: an order
// statistic that is such a bound with overwhelming probability only -- the refine kernel VERIFIES it (flag 16).
cudaError_t launch_sample_threshold(cudaStream_t st, const void* sample, int64_t sample_rows, int b, int rank, const float* eps,
                                    float* thr);
// One CTA per query: tau~ = kk-th largest coarse candidate; keep candidates with coarse >= tau~ - 2*eps[q]; re-score
// them exactly (fp32, the similarity kernel's summation order); sort; write (score, embeddings.id) x kk.
// flags[q] |= 2 candidate list overflowed, 4 fewer than kk candidates, 8 survivor list overflowed, 16 the filter
// threshold thr[q] turned out ABOVE tau~ - 2*eps[q] (the candidate list may miss rows: only possible with a
// statistical threshold): such queries are left to the caller's exact path.  stats[q] (optional) = survivors re-scored.
// Output layout: entry i of query q goes to scores / keys / ids [q * stride + i] (scores, keys optional), its count
// to counts[q * count_stride].  Two users: plain (b, k) arrays, and the packed per-query records of the sharded
// path ([keys(k) | ids(k) | count], 2k+1 int64 words) whose keys carry GLOBAL rows (row0 + local row).
struct RefineOut {
    float* scores; u64* keys; int64_t* ids; int64_t stride;
    int32_t* counts; int64_t count_stride;
    int cap = 0;     // > 0 (REFINE_PARTIAL records only): ship at most cap entries; bit 30 of count = there were more
};
constexpr int32_t REFINE_COUNT_TRUNCATED = 1 << 30;
// Global scratch of the split refine (batch.cu): survivors' rows and exact keys, [b][REFINE_SURVIVOR_CAP] each, and per
// query the survivor count and the verification count (REFINE_PARTIAL).
struct RefineScratch { uint32_t* rows; u64* keys; int32_t* cnt; int32_t* ver; };
constexpr int REFINE_PARTIAL = 1;     // sharded path, global threshold: < kk local candidates is normal; count word = [count, ver]
constexpr int REFINE_DEFER = 2;       // a flagged query gets count -1 in its record (no host read of the flags in between)
// scratch == nullptr (and mode == 0): the one-kernel variant (also SVSB_REFINE_FUSED=1).
// Batched peer exchange (svsb_batch_peer): the kernel that PRODUCES a rank's contribution -- its sample maxima, then its
// candidate records -- stores it straight into every rank's batch window over NVLink peer memory (dst[p], own window
// included); the last CTA to finish (a device-scope ticket, `done`) fences at system scope and release-stores the batch's
// sequence number into every rank's flag word.  Consumers run behind launch_wait_flags on their own window.
struct BatchPush {
    int world = 0;
    unsigned long long seq = 0;
    void* dst[XCHG_MAX_RANKS];          // this rank's region of rank p's window (slot applied)
    u64* flag[XCHG_MAX_RANKS];          // rank p's flag word for (phase, slot, this rank)
    unsigned int* done = nullptr;       // zero on entry, zero again on exit
};
cudaError_t launch_refine(cudaStream_t st, const float* M, int64_t n, int ld, const int64_t* ids, int64_t row0,
                          const float* Q, int b, int ldq, int k, const u64* cand, const int32_t* cand_cnt, int cand_cap,
                          const float* eps, const float* thr, int32_t* flags, RefineOut out, int32_t* stats,
                          const RefineScratch* scratch = nullptr, int mode = 0,
                          const BatchPush* push = nullptr);   // push: records go to dst[p] + q * out.stride ([keys(out.cap) | ids(out.cap) | count, ver])
// One small CTA: wait until flags[0..world) >= seq (ld.acquire.sys); *status |= 1 if a flag does not arrive within
// timeout_ns.  Kernels enqueued behind it on the stream may read what the peers stored before publishing.
cudaError_t launch_wait_flags(cudaStream_t st, const u64* flags, int world, unsigned long long seq, unsigned long long timeout_ns, int* status);
// Sharded path with a GLOBAL filter threshold: every rank extracts the SAMPLE_TOPX largest values of its own sample
// (top[q][0..SAMPLE_TOPX), descending), the lists are exchanged, and thr[q] = (rank-th largest of the union) - 2 eps[q]
// on every rank (rank <= SAMPLE_TOPX; tops = [world][b][SAMPLE_TOPX]).
constexpr int SAMPLE_TOPX = 32;
cudaError_t launch_sample_top(cudaStream_t st, const void* sample, int64_t sample_rows, int b, float* top,
                              const BatchPush* push = nullptr);   // push: the lists go to dst[p][q][0..32) instead of top
// list_stride: floats between rank l's and rank l+1's lists (b * SAMPLE_TOPX for a packed all-gather result)
cudaError_t launch_union_threshold(cudaStream_t st, const float* tops, int64_t list_stride, int world, int b, int rank, const float* eps,
                                   float* thr);
constexpr int REFINE_FLAG_THRESHOLD_HIGH = 16;

// ---- pairwise top pairs (pairs.cu): global candidate list on top of the coarse pass's pairwise mode --------
// The row shards as the pair kernels see them: global rows [row0[s], row0[s + 1]) are M[s] (leading dimension ld) and
// ids[s], peer pointers where the shard lives on another device.  One entry on a single-device engine.
struct PairRows {
    int n = 0;
    int64_t row0[XCHG_MAX_RANKS + 1];
    const float* M[XCHG_MAX_RANKS];
    const int64_t* ids[XCHG_MAX_RANKS];
    __host__ __device__ int shard_of(int64_t r) const { int s = 0; while (s + 1 < n && r >= row0[s + 1]) ++s; return s; }
};
// Sort keys[0..np2) descending; np2 a power of two >= 2048 (pad with 0).
cudaError_t launch_sort_keys_desc(cudaStream_t st, u64* keys, int64_t np2);
cudaError_t launch_pairs_fill_thr(cudaStream_t st, float* thr, int b_pad, int b, const float* scalar);
// query q of the block is global row q_row0 + q, matrix row r global row m_row0 + r; pairs go in as (smaller, larger) row.
// state[0] = entries in the list, state[1] = error flags (1: a per-query list overflowed, 2: the pair list overflowed)
cudaError_t launch_pairs_gather(cudaStream_t st, const u64* cand, const int32_t* cand_cnt, int cand_cap, int b, int64_t q_row0,
                                int64_t m_row0, uint32_t* list_o, u64* list_pair, int64_t list_cap, unsigned long long* state);
// *thr_scalar = max(*thr_scalar, n-th largest coarse score - eps2) over the list (vals == nullptr) or a raw sample
cudaError_t launch_pairs_tau(cudaStream_t st, const uint32_t* list_o, const void* vals /*fp16 sample*/, int64_t vals_count,
                             const unsigned long long* state, int64_t list_cap, int n, float eps2, float* thr_scalar);
cudaError_t launch_pairs_compact(cudaStream_t st, int device, const uint32_t* src_o, const u64* src_pair, const unsigned long long* src_state,
                                 int64_t list_cap, uint32_t* dst_o, u64* dst_pair, unsigned long long* dst_state, const float* thr_scalar);
cudaError_t launch_pairs_sortkeys(cudaStream_t st, const u64* list_pair, int64_t count, int64_t np2, u64* keys);
cudaError_t launch_pairs_rescore(cudaStream_t st, int device, const PairRows& rows, int ld, const u64* keys, int64_t count, float* scores);
cudaError_t launch_pairs_emit(cudaStream_t st, const int64_t* sel, int64_t k, const u64* keys, const int64_t* ids, int64_t* out_a, int64_t* out_b);
// Merge n_lists pair lists (list l at [l * stride ..), counts[l] valid), each sorted by (score desc, row a asc, row b asc)
// with no pair in two lists, into the top k under the same order (select.cu); rows become embeddings.ids through rows.ids.
cudaError_t launch_merge_sorted_pairs(cudaStream_t st, const float* scores, const int64_t* rows_a, const int64_t* rows_b,
                                      const int32_t* counts, int n_lists, int64_t stride, int64_t k, const PairRows& rows,
                                      float* out_scores, int64_t* out_a, int64_t* out_b, int32_t* out_count);

int sm_count(int device);
inline int64_t next_pow2(int64_t v) { int64_t p = 1; while (p < v) p <<= 1; return p; }

}  // namespace svsb
