// Internal structures of the engine (engine.cu) shared with the subsystems that live in their own files:
// multi.cu (several devices in one process), mutate.cu (incremental updates), loader.cu (native SQLite scan).
#pragma once
#include "../../include/svsb200.h"
#include "kernels.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

using namespace svsb;

// ------------------------------------------------------------------------------------------------
// errors, launch counter
// ------------------------------------------------------------------------------------------------
extern thread_local std::string g_err;
static inline int env_int(const char* name, int dflt) { const char* s = getenv(name); return s ? atoi(s) : dflt; }
extern std::atomic<int64_t> g_launches;

static inline int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            (void)cudaGetLastError();                                                              \
            return fail(_e == cudaErrorMemoryAllocation ? SVSB_E_NOMEM : SVSB_E_CUDA,              \
                        std::string(#call) + ": " + cudaGetErrorString(_e));                       \
        }                                                                                          \
    } while (0)

// ------------------------------------------------------------------------------------------------
// data structures
// ------------------------------------------------------------------------------------------------
// Device memory of one shard.  Shared by the generations of one lineage: an incremental update (svsb_apply_mutations)
// publishes a NEW generation that appends rows behind the old generation's last row in the same buffers, so the old
// generation -- and the in-flight queries that pin it -- keeps reading exactly the rows it had.
struct ShardBuf {
    int dev = 0;
    float* M = nullptr;          // cap_rows x ld floats
    int64_t* ids = nullptr;      // cap_rows
    int64_t cap_rows = 0;
    // fp16 shadow M16 = fp16(M * 2^12), cap_rows x ld16 halfs (DESIGN.md section 6): rows [0, m16_rows) are converted.
    // Built at load for the single-query filter when it fits, else lazily by the first batch; appended rows are
    // converted by the update that writes them (shadow_sync).
    std::mutex m16_mu;
    void* M16 = nullptr; int ld16 = 0; int64_t m16_rows = 0;
    // int8 shadow for the single-query int8 filter (DESIGN.md section 4, K1f8), one allocation: M8 = cap_rows x ld8 bytes,
    // then s8 = cap_rows scales, then e8 = the error word E (only raised).  Built next to M16 by filter_attach when it fits,
    // rows [0, m8_rows) converted; guarded by m16_mu.
    void* M8 = nullptr; float* s8 = nullptr; float* e8 = nullptr; int ld8 = 0; int64_t m8_rows = 0;
    ~ShardBuf() {
        if (M || ids || M16 || M8) cudaSetDevice(dev);
        if (M) cudaFree(M);
        if (ids) cudaFree(ids);
        if (M16) cudaFree(M16);
        if (M8) cudaFree(M8);
    }
};

struct Shard {
    int dev = 0;
    int64_t row0 = 0, n = 0;     // n = rows of the buffer this generation uses (physical rows, tombstoned ones included)
    float* M = nullptr;          // == buf->M, buf->ids (raw copies for the hot path)
    int64_t* ids = nullptr;
    std::shared_ptr<ShardBuf> buf;
    // tombstones (svsb_apply_mutations): one byte per physical row, 1 = live; null = every row is live.  Owned by the
    // generation (a delete must not disturb queries still running on the previous generation).
    uint8_t* live = nullptr;
    int64_t n_live = 0;
    // == buf->M16 when this view's single queries take the fp16 filter (set before the generation is published, never
    // changed after; null: K1 -- see filter_shadow in engine.cu)
    const void* M16 = nullptr;
    // == buf->M8 when the int8 filter is available to this view as well (set with M16)
    const void* M8 = nullptr;
};

struct Generation {
    uint64_t id = 0;
    int64_t n = 0;               // physical rows over all shards
    int64_t n_live = 0;          // rows a query can return (== n unless rows were tombstoned)
    int d = 0, ld = 0;
    int norm_mode = SVSB_NORM_CHECK;
    bool owns_live = true;       // false for the per-device views of a multi-device generation (child_gen)
    std::vector<Shard> shards;
    float max_dev = 0.f;
    int64_t n_out_of_tol = 0;
    // multi-device engines: one single-shard view per device, what that device's shard engine queries
    std::vector<std::shared_ptr<Generation>> child_gen;
    // fp16 shadow of shard 0 for the batched coarse contraction (shard 0's buf->M16 once ensure_m16 has covered its rows)
    std::mutex m16_mu;
    void* M16 = nullptr; int ld16 = 0;
    // set once a batch saw its statistical filter thresholds fail verification (rows not in random order w.r.t. the
    // queries): later batches of this generation use the guaranteed thresholds
    std::atomic<bool> batch_guaranteed{false};
    bool has_tombstones() const { return n_live != n; }
    ~Generation() {
        child_gen.clear();
        if (owns_live)
            for (auto& s : shards) if (s.live) { cudaSetDevice(s.dev); cudaFree(s.live); }
    }
};

// per-device scratch for one in-flight query
struct svsb_workspace {
    int dev = 0;
    cudaStream_t st = nullptr;       // owned when created by the engine; null for the stateless API
    bool own_stream = false;
    float* d_q = nullptr;   int q_cap = 0;
    float* scores = nullptr; int64_t n_cap = 0;
    u64* gmax = nullptr;     int64_t g_cap = 0;
    u64* cand = nullptr;     int64_t cand_cap = 0;
    u64* sortbuf = nullptr;  int64_t sort_cap = 0;
    u64* out_keys = nullptr; float* out_scores = nullptr; int64_t* out_ids = nullptr; int64_t out_cap = 0;
    int32_t* out_count = nullptr;
    uint32_t* fstate = nullptr;      // fp16 filter: candidate threshold + rows re-scored (launch_filter_refine)
    u64* mscr_keys = nullptr; int64_t* mscr_ids = nullptr; int64_t mscr_cap = 0;   // merge scratch
    cudaEvent_t ev = nullptr, ev0 = nullptr, ev1 = nullptr, ev_sel = nullptr;
    // The similarity kernel leaves group maxima in gmax and only a SUCCESSFUL selection kernel re-zeroes them
    // (select.cu).  Set before the similarity launch, cleared once the selection is enqueued: a call that failed in
    // between leaves it set and the next user of this (pooled) workspace re-zeroes gmax first.
    bool gmax_dirty = false;

    int ensure_rows(int64_t n) {
        cudaSetDevice(dev);
        if (gmax_dirty && gmax && n <= n_cap) {
            CU(cudaMemset(gmax, 0, (size_t)g_cap * 8));
            CU(cudaStreamSynchronize(cudaStreamLegacy));
            gmax_dirty = false;
        }
        if (n > n_cap) {
            if (scores) cudaFree(scores); if (gmax) cudaFree(gmax); if (cand) cudaFree(cand);
            scores = nullptr; gmax = nullptr; cand = nullptr; n_cap = 0;
            const int shift = group_shift_for(n);
            const int64_t G = (n + ((int64_t)1 << shift) - 1) >> shift;
            int64_t cc = (int64_t)K_FAST_MAX << shift; if (cc > n) cc = n;
            cc += K_FAST_MAX;                       // room for the overflow path to re-home the sort buffer
            CU(cudaMalloc(&scores, (size_t)n * 4));
            CU(cudaMalloc(&gmax, (size_t)G * 8));
            CU(cudaMemset(gmax, 0, (size_t)G * 8));
            // cudaMemset runs on the legacy default stream, asynchronously to the host, and the engine's streams are
            // non-blocking: without this wait a similarity kernel could write group maxima BEFORE the zeroing lands
            CU(cudaStreamSynchronize(cudaStreamLegacy));
            CU(cudaMalloc(&cand, (size_t)cc * 8));
            n_cap = n; g_cap = G; cand_cap = cc; gmax_dirty = false;
        }
        return SVSB_OK;
    }
    int ensure_q(int ld) {
        cudaSetDevice(dev);
        if (ld > q_cap) { if (d_q) cudaFree(d_q); d_q = nullptr; CU(cudaMalloc(&d_q, (size_t)ld * 4)); q_cap = ld; }
        return SVSB_OK;
    }
    int ensure_out(int64_t k) {
        cudaSetDevice(dev);
        if (!out_count) CU(cudaMalloc(&out_count, 64));
        if (!fstate) CU(cudaMalloc(&fstate, 8));
        if (k > out_cap) {
            if (out_keys) cudaFree(out_keys); if (out_scores) cudaFree(out_scores); if (out_ids) cudaFree(out_ids);
            out_keys = nullptr; out_scores = nullptr; out_ids = nullptr; out_cap = 0;
            CU(cudaMalloc(&out_keys, (size_t)k * 8));
            CU(cudaMalloc(&out_scores, (size_t)k * 4));
            CU(cudaMalloc(&out_ids, (size_t)k * 8));
            out_cap = k;
        }
        return SVSB_OK;
    }
    int ensure_sort(int64_t n) {
        cudaSetDevice(dev);
        int64_t need = next_pow2(n); if (need < 2048) need = 2048;
        if (need > sort_cap) {
            if (sortbuf) cudaFree(sortbuf);
            sortbuf = nullptr; sort_cap = 0;                // a failed allocation leaves no capacity behind
            CU(cudaMalloc(&sortbuf, (size_t)need * 8));
            sort_cap = need;
        }
        return SVSB_OK;
    }
    int ensure_merge_scratch(int64_t entries) {
        cudaSetDevice(dev);
        if (entries > mscr_cap) {
            if (mscr_keys) cudaFree(mscr_keys); if (mscr_ids) cudaFree(mscr_ids);
            mscr_keys = nullptr; mscr_ids = nullptr; mscr_cap = 0;
            CU(cudaMalloc(&mscr_keys, (size_t)entries * 8));
            CU(cudaMalloc(&mscr_ids, (size_t)entries * 8));
            mscr_cap = entries;
        }
        return SVSB_OK;
    }
    void release() {
        cudaSetDevice(dev);
        void* ptrs[] = {d_q, scores, gmax, cand, sortbuf, out_keys, out_scores, out_ids, out_count, fstate, mscr_keys, mscr_ids};
        for (void* p : ptrs) if (p) cudaFree(p);
        if (ev) cudaEventDestroy(ev); if (ev0) cudaEventDestroy(ev0); if (ev1) cudaEventDestroy(ev1);
        if (ev_sel) cudaEventDestroy(ev_sel);
        if (own_stream && st) cudaStreamDestroy(st);
    }
};
typedef svsb_workspace DevWs;

struct QueryCtx {
    std::vector<DevWs> ws;                 // one per engine device
    std::unique_ptr<DevWs> alt;            // second buffer set + the selection stream of the pipelined bench loop (device 0)
    DevWs* last = nullptr;                 // workspace holding the last single-device bench result
    // pinned host staging
    float* h_q = nullptr; int h_q_cap = 0;
    float* h_scores = nullptr; int64_t* h_ids = nullptr; int32_t* h_count = nullptr; int64_t h_out_cap = 0;
    // device-0 gather + merge outputs (multi-device)
    u64* g_keys = nullptr; int64_t* g_ids = nullptr; int32_t* g_counts = nullptr; int64_t g_stride = 0;
    float* m_scores = nullptr; int64_t* m_ids = nullptr; int32_t* m_count = nullptr; int64_t m_cap = 0;
    cudaEvent_t ev_merge = nullptr; bool merge_recorded = false;   // last merge that read g_keys / g_ids
    cudaEvent_t ev_gemv = nullptr;         // svsb_query_submit: this context's similarity pass has finished
};

struct Slab {
    float* rows = nullptr; int64_t* ids = nullptr;
    std::vector<cudaEvent_t> ev;           // per device: last copy out of this slab
    std::vector<char> pending;
};

struct Loading {
    std::shared_ptr<Generation> gen;
    int norm_mode = SVSB_NORM_CHECK;
    int64_t loaded = 0;
    int64_t slab_rows = 0;
    int cur = 0;
    bool borrowed = false;
};

// A block of packed candidate records, one per query (include/svsb200.h, sharded deployment):
// Record layout: 2*cap+1 int64 words = [ keys (cap, uint64: ordered score << 32 | ~global_row) |
//                                        embeddings.id (cap) | count (int32 in the low half of the last word) ].
// The batch records of the global threshold (REFINE_PARTIAL) carry [count, ver] in the last word.
struct RecordView {
    int64_t* base = nullptr;                 // record 0
    int cap = 0;                             // entries per record
    int64_t words() const { return 2 * (int64_t)cap + 1; }
    int64_t* rec(int64_t q) const { return base + q * words(); }
    u64* keys(int64_t q) const { return reinterpret_cast<u64*>(rec(q)); }
    int64_t* ids(int64_t q) const { return rec(q) + cap; }
    int32_t* count(int64_t q) const { return reinterpret_cast<int32_t*>(rec(q) + 2 * (int64_t)cap); }
    RecordView from(int64_t q) const { return {rec(q), cap}; }
    // the refine kernel writing records 0, 1, ...; partial: REFINE_PARTIAL records of at most cap entries.
    // base == null: a BatchPush stores the records into the peers' windows, only the layout is used.
    RefineOut refine_out(bool partial = false) const {
        if (!base) return {nullptr, nullptr, nullptr, words(), nullptr, 2 * words(), partial ? cap : 0};
        return {nullptr, keys(0), ids(0), words(), count(0), 2 * words(), partial ? cap : 0};
    }
    // the multi-query selection writing records 0, 1, ... (its scores go to a separate buffer, score_stride apart)
    SelectStrides select_strides(int64_t score_stride) const {
        SelectStrides s; s.keys = words(); s.oscores = score_stride; s.ids = words(); s.count = 2 * words();
        return s;
    }
};

// Merge [n_lists][batch] records (list l + 1's block starts list_words words after list l's) into [batch][k] outputs.
// sk / sp: merge scratch of batch * n_lists * recs.cap entries, needed only when n_lists * recs.cap > K_FAST_MAX.
// verify_k >= 0: the records carry [count, ver] (REFINE_PARTIAL); status: a batch window's timeout word (or null).
static inline int merge_records(cudaStream_t st, const RecordView& recs, int n_lists, int64_t list_words, int batch, int k, u64* sk,
                                int64_t* sp, float* out_scores, int64_t* out_ids, int32_t* out_counts, int verify_k = -1,
                                const int* status = nullptr) {
    CU(launch_merge_ex(st, recs.keys(0), recs.ids(0), recs.count(0), n_lists, recs.cap, k, batch, list_words, recs.words(),
                       2 * list_words, 2 * recs.words(), sk, sp, out_scores, out_ids, out_counts, verify_k, status));
    return SVSB_OK;
}

// workspace of the batched path: coarse operands, thresholds, candidate lists, outputs (device) + pinned staging
struct BatchWs {
    int dev = 0;
    cudaStream_t st = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    // capacities
    int cap_b = 0, cap_ld = 0, cap_k = 0; int64_t cap_sample = 0; int cand_cap = 0;
    float* dQ = nullptr; void* dQ16 = nullptr;
    float* eps = nullptr; float* thr = nullptr; int32_t* flags = nullptr; int32_t* cand_cnt = nullptr; int32_t* stats = nullptr;
    float* sample = nullptr; u64* cand = nullptr;
    RefineScratch rs = {nullptr, nullptr, nullptr, nullptr};     // split refine: survivors' rows / exact keys / counts
    float* tops = nullptr;                                        // [cap_b][SAMPLE_TOPX]: this rank's largest sample values (sharded path)
    uint64_t global_gen = 0; int global_b = 0, global_k = 0;      // svsb_batch_sample_tops -> svsb_batch_global_records hand-over
    float* o_scores = nullptr; int64_t* o_ids = nullptr; int32_t* o_counts = nullptr;
    float* h_Q = nullptr; float* h_scores = nullptr; int64_t* h_ids = nullptr; int32_t* h_counts = nullptr;
    int32_t* h_flags = nullptr; int32_t* h_stats = nullptr; int32_t* h_cnt = nullptr;

    void release_device() {
        cudaSetDevice(dev);
        void* ptrs[] = {dQ, dQ16, eps, thr, flags, cand_cnt, stats, sample, cand, o_scores, o_ids, o_counts,
                        rs.rows, rs.keys, rs.cnt, rs.ver, tops};
        for (void* p : ptrs) if (p) cudaFree(p);
        void* hp[] = {h_Q, h_scores, h_ids, h_counts, h_flags, h_stats, h_cnt};
        for (void* p : hp) if (p) cudaFreeHost(p);
        dQ = nullptr; dQ16 = nullptr; eps = thr = nullptr; flags = cand_cnt = stats = nullptr; sample = nullptr; cand = nullptr;
        o_scores = nullptr; o_ids = nullptr; o_counts = nullptr;
        rs = {nullptr, nullptr, nullptr, nullptr}; tops = nullptr;
        h_Q = h_scores = nullptr; h_ids = nullptr; h_counts = h_flags = h_stats = h_cnt = nullptr;
        cap_b = cap_ld = cap_k = 0; cap_sample = 0; cand_cap = 0;
    }
    void release() {
        release_device();
        for (auto& e : ev) if (e) { cudaEventDestroy(e); e = nullptr; }
        if (st) { cudaStreamDestroy(st); st = nullptr; }
    }
};

// workspace of the small-batch exact path (gemv_tma_mq_kernel + one selection CTA per query)
struct MqWs {
    int dev = 0;
    cudaStream_t st = nullptr;
    int cap_b = 0, cap_ld = 0; int64_t cap_n = 0, G = 0, cand_cap = 0, cap_out = 0;
    float* dQ = nullptr; float* scores = nullptr; u64* gmax = nullptr; u64* cand = nullptr;
    u64* o_keys = nullptr; float* o_scores = nullptr; int64_t* o_ids = nullptr; int32_t* o_counts = nullptr;
    float* h_Q = nullptr;
    bool gmax_dirty = false;

    int ensure(int b, int64_t n, int ld, int64_t k) {
        cudaSetDevice(dev);
        if (!st) CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        if (b > cap_b || n > cap_n) {
            CU(cudaStreamSynchronize(st));
            const int nb = std::max(b, cap_b); const int64_t nn = std::max(n, cap_n);
            void* ptrs[] = {scores, gmax, cand, o_counts};
            for (void* p : ptrs) if (p) cudaFree(p);
            scores = nullptr; gmax = nullptr; cand = nullptr; o_counts = nullptr; cap_b = 0; cap_n = 0;
            const int shift = group_shift_for(nn);
            G = (nn + ((int64_t)1 << shift) - 1) >> shift;
            cand_cap = std::min<int64_t>((int64_t)K_FAST_MAX << shift, nn) + K_FAST_MAX;
            CU(cudaMalloc(&scores, (size_t)nb * nn * 4));
            CU(cudaMalloc(&gmax, (size_t)nb * G * 8));
            CU(cudaMalloc(&cand, (size_t)nb * cand_cap * 8));
            CU(cudaMalloc(&o_counts, (size_t)nb * 4));
            cap_b = nb; cap_n = nn; gmax_dirty = true; cap_out = 0; cap_ld = 0;
        }
        if (gmax_dirty) {
            CU(cudaMemsetAsync(gmax, 0, (size_t)cap_b * G * 8, st));
            gmax_dirty = false;
        }
        if (ld > cap_ld) {
            CU(cudaStreamSynchronize(st));
            if (dQ) cudaFree(dQ);
            if (h_Q) cudaFreeHost(h_Q);
            dQ = nullptr; h_Q = nullptr; cap_ld = 0;
            CU(cudaMalloc(&dQ, (size_t)cap_b * ld * 4));
            CU(cudaMallocHost(&h_Q, (size_t)cap_b * ld * 4));
            cap_ld = ld;
        }
        if ((int64_t)cap_b * k > cap_out) {
            CU(cudaStreamSynchronize(st));
            void* ptrs[] = {o_keys, o_scores, o_ids};
            for (void* p : ptrs) if (p) cudaFree(p);
            o_keys = nullptr; o_scores = nullptr; o_ids = nullptr; cap_out = 0;
            const int64_t e = (int64_t)cap_b * k;
            CU(cudaMalloc(&o_keys, (size_t)e * 8));
            CU(cudaMalloc(&o_scores, (size_t)e * 4));
            CU(cudaMalloc(&o_ids, (size_t)e * 8));
            cap_out = e;
        }
        return SVSB_OK;
    }
    void release() {
        cudaSetDevice(dev);
        void* ptrs[] = {dQ, scores, gmax, cand, o_keys, o_scores, o_ids, o_counts};
        for (void* p : ptrs) if (p) cudaFree(p);
        if (h_Q) cudaFreeHost(h_Q);
        if (st) cudaStreamDestroy(st);
    }
};

// Other ranks' memory as the one-process-per-GPU deployment reaches it (engine.cu "peer memory"): the CUDA IPC mappings
// a rank opened, and peer access to the devices of this process.
struct PeerMaps {
    std::vector<void*> opened;
    int open(const void* handle, void** out, const char* who);   // a peer's 64-byte cudaIpcMemHandle_t
    int reach(int self, int dev, const char* who);                // device self (the current one) -> device dev's memory
    void close();
};

// What the gather window (Xchg) and the batch window (BXchg) share.
struct PeerWindow {
    int world = 0, rank = 0;
    unsigned char* block = nullptr;
    std::vector<unsigned char*> peer_block;              // per rank (own entry = block)
    PeerMaps maps;
    bool connected = false;
    unsigned long long seq = 0;
    unsigned long long timeout_ns = 30ull * 1000000000ull;   // a wait kernel gives up on a peer (SVSB_XCHG_TIMEOUT_MS)
    int publish(void* handle_out);                       // the end of a create; handle_out: this window's IPC handle
    int connect(const void* handles, const char* who);   // world x 64-byte IPC handles in rank order
    // windows of engines in this process; window_of(peer, this) = the peer's window if it matches this one, else null
    int connect_local(int dev, svsb_engine* const* engines, PeerWindow* (*window_of)(svsb_engine*, const PeerWindow*), const char* who);
    void unmap();                                        // back to the state publish left
};

// Batch window of the one-process-per-GPU deployment (svsb_bxchg_*, svsb_batch_peer): per slot and source rank a region
// for the rank's sample maxima and one for its candidate records, written by the peers' kernels over NVLink peer memory.
//   [flags: 2 phases x slots x world u64, padded to 256 B][tops: slots x world x B_MAX x 32 f32][records: slots x world x B_MAX x (2 rec_cap + 1) i64]
struct BXchg : PeerWindow {
    static constexpr int SLOTS = 2, B_MAX = COARSE_MAX_BATCH;
    int rec_cap = 0;
    size_t flags_bytes = 0, tops_bytes = 0, bytes = 0;
    unsigned int* done = nullptr;            // two last-block tickets (sample maxima, records)
    int* status = nullptr;                   // device word: 1 = a wait timed out
    // svsb_batch_peer with flag bit 0: the verifying merge of batch j is enqueued behind the FIRST phase of batch j+1 (or by
    // svsb_batch_peer_flush), so the peers have that long to deliver their records before this rank's stream waits for them
    struct Deferred {
        bool pending = false;
        int slot = 0, rec_cap = 0, k = 0, b = 0; unsigned long long seq = 0;
        float* out_scores = nullptr; int64_t* out_ids = nullptr; int32_t* out_counts = nullptr;
    } deferred;
    int64_t tops_region() const { return (int64_t)B_MAX * SAMPLE_TOPX; }                       // floats per (slot, source)
    int64_t rec_region() const { return (int64_t)B_MAX * (2 * (int64_t)rec_cap + 1); }         // words per (slot, source)
    u64* flag(unsigned char* blk, int phase, int slot, int src) const { return reinterpret_cast<u64*>(blk) + ((int64_t)phase * SLOTS + slot) * world + src; }
    float* tops(unsigned char* blk, int slot, int src) const { return reinterpret_cast<float*>(blk + flags_bytes) + ((int64_t)slot * world + src) * tops_region(); }
    int64_t* recs(unsigned char* blk, int slot, int src) const { return reinterpret_cast<int64_t*>(blk + flags_bytes + tops_bytes) + ((int64_t)slot * world + src) * rec_region(); }
};

// Peer exchange of the one-process-per-GPU deployment (kernels.cuh "peer exchange"): this rank's gather window,
// the peers' windows opened over CUDA IPC (or plain pointers inside one process), and a synchronous query context.
// block = [flags: slots*world u64, padded to 256 B][window]
struct Xchg : PeerWindow {
    int cap = 0, slots = 4;
    int64_t rec_words = 0;
    size_t flags_bytes = 0;
    // Pipelined path: the merge of query j is enqueued on the side stream BEHIND the selection of query j+1, so a
    // peer has a whole query time to deliver its record before this rank's side stream would wait for it.
    struct DeferredMerge {
        bool pending = false;
        int slot = 0, k = 0; unsigned long long seq = 0;
        u64* sk = nullptr; int64_t* sp = nullptr;
        float* out_scores = nullptr; int64_t* out_ids = nullptr; int32_t* out_count = nullptr;
        cudaEvent_t ev_done = nullptr;                   // recorded behind the merge once it is enqueued (submit / wait tickets)
    } deferred;
    // svsb_query_peer_submit / _wait: host-buffer queries with several in flight.  A ticket owns its pinned query and
    // result buffers and a device copy of the query (the next query is staged while this one's similarity pass runs).
    struct Ticket {
        float* h_q = nullptr; float* d_q = nullptr;
        float* h_scores = nullptr; int64_t* h_ids = nullptr; int32_t* h_count = nullptr;
        cudaEvent_t ev = nullptr;
        bool busy = false; int k = 0; unsigned long long seq = 0;
    };
    static constexpr int N_TICKETS = 3;
    Ticket tk[N_TICKETS];
    int tk_ld = 0, tk_next = 0;
    // measurement aid (SVSB_XCHG_STAMPS=1): %globaltimer stamps of the last STAMP_RING synchronous peer queries --
    // selection kernel phases (16 words) + merge kernel (24 words) per query
    static constexpr int STAMP_RING = 1024, STAMP_WORDS = 40;
    u64* stamps = nullptr;
    cudaEvent_t ev_join = nullptr;
    // synchronous path (svsb_query_peer): own stream, device query, pinned staging; results land in pinned
    // host memory straight from the merge kernel (mapped, no copy back)
    cudaStream_t st = nullptr;
    DevWs ws;
    float* h_q = nullptr; int h_q_cap = 0;
    float* h_scores = nullptr; int64_t* h_ids = nullptr; int32_t* h_count = nullptr; int64_t h_cap = 0;
    u64* flags_of(unsigned char* b, int slot) const { return reinterpret_cast<u64*>(b) + (size_t)slot * world; }
    u64* rec_of(unsigned char* b, int slot, int src) const {
        return reinterpret_cast<u64*>(b + flags_bytes) + ((size_t)slot * world + src) * rec_words;
    }
};

// The fp16 shadow of one shard as a rectangle task of the pair search copies blocks of it.  dev >= 0: memory of that
// device of this process (cudaMemcpyPeerAsync names it by ordinal).  dev < 0: a pointer the copying device's context
// addresses directly -- a CUDA IPC mapping of another process's shard, or a peer engine's memory in this process; it
// is copied with cudaMemcpyAsync (device ordinals are per process, so they cannot name another process's device).
struct PairShadow { const void* M16 = nullptr; int dev = -1; };

// Pair search of the one-process-per-GPU deployment (svsb_pairs_*): the generation this rank exported (pinned: the peers
// map its buffers) and, once connected, every rank's shard as the pair kernels address it.
struct PairsShard {
    std::shared_ptr<Generation> gen;
    int world = 0, rank = 0, d = 0;
    bool connected = false;
    std::vector<int64_t> shard_rows;                     // per rank
    std::vector<PairShadow> shadows;                     // per rank
    PairRows rows;                                       // global rows, counted from rank 0's first row
    PeerMaps maps;
    cudaEvent_t ev = nullptr;                            // the caller's stream -> the pass's stream
};

struct svsb_engine {
    std::vector<int> devs;
    std::mutex mu;                          // guards current, loading, pool bookkeeping
    std::condition_variable cv;
    std::shared_ptr<Generation> current;
    uint64_t next_gen = 1;
    std::unique_ptr<Loading> loading;
    std::vector<Slab> slabs; int64_t slab_bytes_rows = 0, slab_ids_cap = 0;
    std::vector<cudaStream_t> copy_st;      // per device
    std::vector<std::unique_ptr<QueryCtx>> pool_free;
    int ctx_total = 0, ctx_max = 4;
    // svsb_query_submit keeps several contexts in flight.  Their similarity passes all go down ONE stream, back to back
    // (pass j+1 starts when pass j ends, so the one SM each pass leaves free really is free for the single-CTA
    // selections, which run on the contexts' own streams) -- the structure of the device-resident pipelined loop.
    std::mutex chain_mu;
    cudaStream_t submit_st = nullptr;
    // batched path (one batch at a time)
    std::mutex batch_mu;
    std::unique_ptr<struct BatchWs> batch_ws;
    std::unique_ptr<MqWs> mq_ws;            // small exact batches (guarded by batch_mu as well)
    // bench state
    std::vector<float*> bench_q; int bench_nq = 0, bench_d = 0, bench_ld = 0;
    std::unique_ptr<QueryCtx> bench_ctx;
    std::vector<cudaEvent_t> bench_kev;                  // similarity-kernel timing events of svsb_bench_run (device 0)
    int bench_route = 0;                                 // the last svsb_bench_run's route: 0 K1, 16 / 8 the fp16 / int8 filter
    // sharded deployment (one process per GPU)
    int64_t shard_row0 = 0;                              // global row of this engine's first row
    std::vector<std::unique_ptr<DevWs>> shard_ws;        // workspaces for svsb_enqueue_local_topk (by slot)
    std::vector<cudaEvent_t> kev; size_t kev_used = 0;   // similarity-kernel timing events
    cudaStream_t side_st = nullptr;                      // selection kernels of the pipelined sharded path
    std::vector<char> sel_pending;                       // per slot: a selection is (or was) in flight on side_st
    std::unique_ptr<Xchg> xchg;
    std::unique_ptr<BXchg> bxchg;
    std::unique_ptr<PairsShard> pairs;
    // several devices in ONE process (svsb_create with n_dev > 1, multi.cu): one shard engine per device, driven by one
    // worker thread each, candidate records pushed into device 0's gather window by the selection kernels
    struct Multi* multi = nullptr;
    bool is_kid = false;                                 // a per-device shard engine owned by a multi-device engine
    std::mutex mutate_mu;                                // one svsb_apply_mutations / load publication at a time
};

static inline int round_up4(int d) { return (d + 3) & ~3; }

// host queries Q[b][d] -> dst[b][ld], zero padded to the rows' leading dimension (staging of the batched paths)
static inline void stage_queries(float* dst, const float* Q, int b, int d, int ld) {
    for (int i = 0; i < b; ++i) {
        memcpy(dst + (size_t)i * ld, Q + (size_t)i * d, (size_t)d * 4);
        std::fill(dst + (size_t)i * ld + d, dst + (size_t)(i + 1) * ld, 0.f);
    }
}

// a query handle that keeps "the arrays it fetched" alive across an invalidate (svsb_snapshot_*)
struct svsb_snapshot { std::shared_ptr<Generation> gen; };

// ------------------------------------------------------------------------------------------------
// internal interfaces between engine.cu and the subsystem files
// ------------------------------------------------------------------------------------------------
std::shared_ptr<Generation> pin(svsb_engine* e);
int prepare_ws(DevWs& w, const Generation* g, const Shard& s, int64_t kk);
// Convert rows [buf->m16_rows, s.n) of the shard's fp16 shadow (rows from `fresh_from` on were (re)written: they are
// converted again).  No shadow yet: create = 0 leaves it so (*out = null), 1 allocates it when the device keeps ample
// room after it (else *out = null, not an error), 2 allocates it or fails.  The int8 shadow (ShardBuf::M8) is kept the
// same way when it exists; create = 1 also allocates it, under the same room rule, for rows of ld <= FILTER_MAX_LD.
int shadow_sync(const Shard& s, int ld, int64_t fresh_from, int create, cudaStream_t st, void** out);
int engine_create(const int* device_ids, int n_dev, bool as_kid, svsb_engine** out);
int alloc_generation(svsb_engine* e, int64_t n, int d, std::shared_ptr<Generation>& out);
int finish_generation(svsb_engine* e, Generation* g, int norm_mode);
// publish `g` as the engine's resident generation (assigns the id; builds the per-device views of a multi-device engine)
int publish_generation(svsb_engine* e, const std::shared_ptr<Generation>& g, uint64_t* generation);
// local top-k records [b][2k+1] of b device-resident queries on `st` (engine.cu; the body of svsb_batch_local_records)
int batch_local_records_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, cudaStream_t st, const float* d_Q, int32_t b,
                            int32_t k, int64_t* d_records, int32_t* n_fallback);

// pairwise top pairs (engine.cu): one device's share of the pass, in the phases multi.cu runs on every device in turn
// so that all allocations happen before any cross-device work is enqueued
struct DevBufs {                                  // frees everything it handed out
    int dev = 0; std::vector<void*> ptrs;
    DevBufs() = default;
    DevBufs(const DevBufs&) = delete;
    DevBufs& operator=(const DevBufs&) = delete;
    ~DevBufs() { if (ptrs.empty()) return; cudaSetDevice(dev); for (void* p : ptrs) cudaFree(p); }
    template <class T> cudaError_t get(T** out, size_t count) {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) { ptrs.push_back(p); *out = reinterpret_cast<T*>(p); }
        return e;
    }
};
// A task of device `self`: its own shard's rows [m0, m1) against rows [q0, q1) of shard `peer`, every combination
// (peer != self); or, with peer == self, the upper triangle of its whole shard.
struct PairTask { int peer = 0; int64_t m0 = 0, m1 = 0, q0 = 0, q1 = 0; };
std::vector<std::vector<PairTask>> pairs_plan(const std::vector<int64_t>& shard_rows);
// The shards of single-shard views (one per device, scan order) as the pair kernels address them; rows are counted
// from the first view's first row.
PairRows pair_rows_of(const std::vector<Generation*>& views);
struct PairsDev {
    Generation* g = nullptr;                       // this device's single-shard view
    BatchWs* w = nullptr;                          // its batch workspace (stream, thresholds, candidate lists, Q staging); null: no rows
    cudaStream_t st = nullptr;
    DevBufs bufs;
    int64_t n = 0;                                 // pairs asked for
    float eps2 = 0.f;
    int ld16 = 0, cand_cap = 0, s_tiles = 0, tile_stride = 1; int64_t sample_rows = 0; bool bootstrap = false;
    int64_t LC = 0;                                // pair list capacity
    uint32_t* lo[2] = {nullptr, nullptr}; u64* lp[2] = {nullptr, nullptr}; unsigned long long* lstate[2] = {nullptr, nullptr};
    float* thr = nullptr;                          // the device's running threshold
    int cur = 0;
    int64_t C = 0;                                 // pairs in the list after the coarse pass
    int64_t kl = 0;                                // entries of the device's result list: min(n, C)
    int64_t np2 = 0; int shift = 0;
    u64* keys = nullptr; float* scores = nullptr; u64* sortbuf = nullptr; u64* gmax = nullptr;
    u64* o_keys = nullptr; float* o_scores = nullptr; int64_t* o_sel = nullptr; int32_t* o_cnt = nullptr;
    int64_t* o_a = nullptr; int64_t* o_b = nullptr;
};
// threshold margin (2 eps) of the fp16 coarse pair score for d components and rows of norm at most R
float pairs_eps2(int d, float R);
// workspace, fp16 shadow of the shard, pair lists (sizes fixed by n)
int pairs_dev_prepare(svsb_engine* e, Generation* g, int64_t n, float eps2, PairsDev& r);
// coarse filter over the device's tasks with its own running threshold; synchronises the device's stream, sets r.C.
// shadows[s]: shard s's fp16 rows (read only by rectangle tasks against shard s)
int pairs_dev_coarse(PairsDev& r, int self, const std::vector<PairTask>& tasks, const std::vector<PairShadow>& shadows, const PairRows& rows);
// buffers sized by r.C
int pairs_dev_alloc(PairsDev& r);
// exact re-score of the list, its top r.kl in the final order: r.o_scores, r.o_a / r.o_b (ids[row], or rows if ids is null)
int pairs_dev_finish(PairsDev& r, const PairRows& rows, const int64_t* ids);

// multi.cu
int  multi_top_pairs(svsb_engine* e, const std::shared_ptr<Generation>& g, int64_t n, float eps2, float* out_scores,
                     int64_t* out_ids_a, int64_t* out_ids_b, int64_t* out_count);
int  multi_create(svsb_engine* e);
void multi_destroy(svsb_engine* e);
int  multi_publish(svsb_engine* e, const std::shared_ptr<Generation>& g);
int  multi_query(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int64_t kk,
                 float* out_scores, int64_t* out_ids, int32_t* out_count);
struct svsb_ticket;
int  multi_submit(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int64_t kk, svsb_ticket** out);
int  multi_wait(svsb_engine* e, svsb_ticket* t, float* out_scores, int64_t* out_ids, int32_t* out_count);
int  multi_query_batch(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* Q, int32_t b, int32_t d, int32_t k,
                       float* out_scores, int64_t* out_ids, int32_t* out_counts);
int  multi_bench_run(svsb_engine* e, const std::shared_ptr<Generation>& g, int32_t k, int32_t iters, float* total_ms, float* gemv_ms);
int  multi_bench_last_result(svsb_engine* e, int32_t k, float* out_scores, int64_t* out_ids, int32_t* out_count);
