// The engine object and the C ABI (include/svsb200.h).
//
// Host-side responsibilities, all replacing pieces of the reference's `_EmbeddingsMatrix`
// (src/svs/kb.py:856-893) and `superheavy()` (src/svs/kb.py:1184-1189, 1622-1627):
//   * generations: the device-resident matrix + embeddings.id table is an immutable, ref-counted
//     snapshot; load builds a new one off to the side and publishes it atomically; invalidate drops
//     the engine's reference; in-flight queries keep theirs (what NumPy refcounts give the reference);
//   * load path: caller rows -> pinned ring slabs -> cudaMemcpyAsync -> row-sharded device matrix with a
//     16-byte-aligned leading dimension -> row-norm kernel;
//   * query contexts: a small pool of {stream, workspace, pinned in/out buffers} per device so that
//     svsb_query is re-entrant from several OS threads;
//   * multi-device: contiguous row shards, per-device GEMV + exact local top-k, candidate lists copied
//     peer-to-peer to device 0 and merged there by one kernel.
#include "engine.cuh"

#include <chrono>

thread_local std::string g_err;
static thread_local bool g_pdl = false;
namespace svsb { void set_pdl(bool on) { g_pdl = on; } bool pdl_enabled() { return g_pdl; } }
std::atomic<int64_t> g_launches{0};
namespace svsb { void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); } }


// ------------------------------------------------------------------------------------------------
// context pool
// ------------------------------------------------------------------------------------------------
static int ctx_create(svsb_engine* e, std::unique_ptr<QueryCtx>& out) {
    std::unique_ptr<QueryCtx> c(new QueryCtx());
    c->ws.resize(e->devs.size());
    for (size_t i = 0; i < e->devs.size(); ++i) {
        DevWs& w = c->ws[i];
        w.dev = e->devs[i];
        CU(cudaSetDevice(w.dev));
        CU(cudaStreamCreateWithFlags(&w.st, cudaStreamNonBlocking));
        w.own_stream = true;
        CU(cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming));
        CU(cudaEventCreate(&w.ev0));
        CU(cudaEventCreate(&w.ev1));
        CU(cudaEventCreateWithFlags(&w.ev_sel, cudaEventDisableTiming));
    }
    out = std::move(c);
    return SVSB_OK;
}
static void ctx_destroy(svsb_engine* e, QueryCtx* c) {
    if (!c) return;
    for (auto& w : c->ws) w.release();
    if (c->alt) c->alt->release();
    if (!e->devs.empty()) cudaSetDevice(e->devs[0]);
    if (c->h_q) cudaFreeHost(c->h_q);
    if (c->h_scores) cudaFreeHost(c->h_scores);
    if (c->h_ids) cudaFreeHost(c->h_ids);
    if (c->h_count) cudaFreeHost(c->h_count);
    if (c->ev_gemv) cudaEventDestroy(c->ev_gemv);
}
// timeout_ms > 0: give up (SVSB_E_STATE) when no context frees up in time -- svsb_query_submit from a caller that already
// holds every context as a pending handle would otherwise wait for itself
static int ctx_acquire(svsb_engine* e, std::unique_ptr<QueryCtx>& out, int timeout_ms = 0) {
    std::unique_lock<std::mutex> lk(e->mu);
    while (true) {
        if (!e->pool_free.empty()) { out = std::move(e->pool_free.back()); e->pool_free.pop_back(); return SVSB_OK; }
        if (e->ctx_total < e->ctx_max) { ++e->ctx_total; break; }
        if (timeout_ms > 0) {
            if (e->cv.wait_for(lk, std::chrono::milliseconds(timeout_ms)) == std::cv_status::timeout && e->pool_free.empty())
                return fail(SVSB_E_STATE, "svsb_query_submit: every query context is pending already (wait for the oldest first)");
        } else e->cv.wait(lk);
    }
    lk.unlock();
    int rc = ctx_create(e, out);
    if (rc != SVSB_OK) { lk.lock(); --e->ctx_total; e->cv.notify_one(); }
    return rc;
}
static void ctx_release(svsb_engine* e, std::unique_ptr<QueryCtx>& c) {
    std::lock_guard<std::mutex> lk(e->mu);
    e->pool_free.push_back(std::move(c));
    e->cv.notify_one();
}
struct CtxLease {
    svsb_engine* e; std::unique_ptr<QueryCtx> c;
    explicit CtxLease(svsb_engine* e_) : e(e_) {}
    ~CtxLease() { if (c) ctx_release(e, c); }
};

static int ctx_ensure_host(QueryCtx* c, int ld, int64_t k) {
    if (ld > c->h_q_cap) { if (c->h_q) cudaFreeHost(c->h_q); c->h_q = nullptr; CU(cudaMallocHost(&c->h_q, (size_t)ld * 4)); c->h_q_cap = ld; }
    if (!c->h_count) CU(cudaMallocHost(&c->h_count, 64));
    if (k > c->h_out_cap) {
        if (c->h_scores) cudaFreeHost(c->h_scores); if (c->h_ids) cudaFreeHost(c->h_ids);
        c->h_scores = nullptr; c->h_ids = nullptr; c->h_out_cap = 0;
        CU(cudaMallocHost(&c->h_scores, (size_t)k * 4));
        CU(cudaMallocHost(&c->h_ids, (size_t)k * 8));
        c->h_out_cap = k;
    }
    return SVSB_OK;
}
// ------------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------------
int engine_create(const int* device_ids, int n_dev, bool as_kid, svsb_engine** out) {
    if (!out) return fail(SVSB_E_INVALID, "svsb_create: out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t ce = cudaGetDeviceCount(&count);
    if (ce != cudaSuccess || count <= 0) {
        (void)cudaGetLastError();
        return fail(SVSB_E_NO_DEVICE, std::string("no CUDA device available (") +
                    (ce != cudaSuccess ? cudaGetErrorString(ce) : "device count 0") + "); svs_b200 has no CPU path");
    }
    std::unique_ptr<svsb_engine> e(new svsb_engine());
    if (!device_ids || n_dev <= 0) e->devs.push_back(0);
    else for (int i = 0; i < n_dev; ++i) {
        if (device_ids[i] < 0 || device_ids[i] >= count) return fail(SVSB_E_INVALID, "svsb_create: device id out of range");
        // duplicates = several "virtual shards" on one GPU: only for testing the multi-shard path on one device
        const char* dup = getenv("SVSB_ALLOW_DUP_DEVICES");
        for (int j = 0; j < i; ++j)
            if (device_ids[j] == device_ids[i] && !(dup && dup[0] == '1'))
                return fail(SVSB_E_INVALID, "svsb_create: duplicate device id");
        e->devs.push_back(device_ids[i]);
    }
    if (const char* s = getenv("SVSB_MAX_CONTEXTS")) { int v = atoi(s); if (v >= 1 && v <= 64) e->ctx_max = v; }
    for (size_t i = 0; i < e->devs.size(); ++i) {
        CU(cudaSetDevice(e->devs[i]));
        int major = 0, minor = 0;
        CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, e->devs[i]));
        CU(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, e->devs[i]));
        if (major != 10) {
            char buf[160];
            snprintf(buf, sizeof buf, "device %d has compute capability %d.%d; svs_b200 is built for sm_100a (B200) only",
                     e->devs[i], major, minor);
            return fail(SVSB_E_NO_DEVICE, buf);
        }
        cudaStream_t st;
        CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
        e->copy_st.push_back(st);
    }
    e->is_kid = as_kid;
    svsb_engine* raw = e.release();
    if (raw->devs.size() > 1) {
        // one shard engine + one worker thread per device, gather windows connected over peer memory (multi.cu)
        int rc = multi_create(raw);
        if (rc != SVSB_OK) { const std::string msg = g_err; svsb_destroy(raw); g_err = msg; return rc; }
    }
    *out = raw;
    return SVSB_OK;
}

extern "C" int svsb_create(const int* device_ids, int n_dev, svsb_t** out) {
    return engine_create(device_ids, n_dev, false, out);
}

static void free_slabs(svsb_engine* e) {
    for (auto& s : e->slabs) {
        if (s.rows) cudaFreeHost(s.rows);
        if (s.ids) cudaFreeHost(s.ids);
        for (auto ev : s.ev) if (ev) cudaEventDestroy(ev);
    }
    e->slabs.clear(); e->slab_bytes_rows = 0; e->slab_ids_cap = 0;
}

static void bxchg_release(svsb_engine* e);
static void pairs_release(svsb_engine* e);
static void xchg_release(svsb_engine* e) {
    Xchg* x = e->xchg.get();
    if (!x) return;
    cudaSetDevice(e->devs[0]);
    if (x->st) cudaStreamSynchronize(x->st);
    x->maps.close();
    if (x->block) cudaFree(x->block);
    if (x->stamps) cudaFree(x->stamps);
    x->ws.release();
    if (x->st) cudaStreamDestroy(x->st);
    if (x->ev_join) cudaEventDestroy(x->ev_join);
    if (x->h_q) cudaFreeHost(x->h_q);
    if (x->h_scores) cudaFreeHost(x->h_scores);
    if (x->h_ids) cudaFreeHost(x->h_ids);
    if (x->h_count) cudaFreeHost(x->h_count);
    for (auto& t : x->tk) {
        if (t.h_q) cudaFreeHost(t.h_q);
        if (t.d_q) cudaFree(t.d_q);
        if (t.h_scores) cudaFreeHost(t.h_scores);
        if (t.h_ids) cudaFreeHost(t.h_ids);
        if (t.h_count) cudaFreeHost(t.h_count);
        if (t.ev) cudaEventDestroy(t.ev);
    }
    e->xchg.reset();
}

extern "C" void svsb_destroy(svsb_t* e) {
    if (!e) return;
    multi_destroy(e);                       // workers joined, shard engines gone, before anything they use is freed
    for (size_t i = 0; i < e->devs.size(); ++i) { cudaSetDevice(e->devs[i]); cudaDeviceSynchronize(); }
    e->loading.reset();
    e->current.reset();
    e->pending.reset();
    for (auto& c : e->pool_free) ctx_destroy(e, c.get());
    e->pool_free.clear();
    if (e->bench_ctx) ctx_destroy(e, e->bench_ctx.get());
    if (e->batch_ws) e->batch_ws->release();
    if (e->mq_ws) e->mq_ws->release();
    for (auto& w : e->shard_ws) if (w) w->release();
    xchg_release(e);
    bxchg_release(e);
    pairs_release(e);
    if (e->side_st) { cudaSetDevice(e->devs[0]); cudaStreamDestroy(e->side_st); }
    if (e->submit_st) { cudaSetDevice(e->devs[0]); cudaStreamDestroy(e->submit_st); }
    for (auto ev : e->kev) cudaEventDestroy(ev);
    if (!e->bench_kev.empty()) { cudaSetDevice(e->devs[0]); for (auto ev : e->bench_kev) cudaEventDestroy(ev); }
    for (size_t i = 0; i < e->bench_q.size(); ++i) if (e->bench_q[i]) { cudaSetDevice(e->devs[i]); cudaFree(e->bench_q[i]); }
    free_slabs(e);
    for (size_t i = 0; i < e->copy_st.size(); ++i) { cudaSetDevice(e->devs[i]); cudaStreamDestroy(e->copy_st[i]); }
    delete e;
}

// ------------------------------------------------------------------------------------------------
// load path
// ------------------------------------------------------------------------------------------------
int alloc_generation(svsb_engine* e, int64_t n, int d, std::shared_ptr<Generation>& out) {
    if (e->has_pending) return fail(SVSB_E_STATE, "a prepared update is pending: svsb_shard_mutations_commit before loading");
    std::shared_ptr<Generation> g(new Generation());
    g->n = n; g->d = d; g->ld = round_up4(d);
    const int64_t nd = (int64_t)e->devs.size();
    const int64_t per = (n + nd - 1) / nd;
    for (int64_t i = 0; i < nd; ++i) {
        Shard s; s.dev = e->devs[i];
        s.row0 = std::min(n, i * per);
        s.n = std::min(n, (i + 1) * per) - s.row0;
        s.row0 += e->shard_row0;                         // keys / synthetic rows are in GLOBAL row numbers
        if (s.n > 0xfffffff0ll) return fail(SVSB_E_INVALID, "more than 2^32 rows per device are not supported");
        g->shards.push_back(s);
    }
    if (n + e->shard_row0 > 0xfffffff0ll) return fail(SVSB_E_INVALID, "more than 2^32 rows in total are not supported");
    g->n_live = n;
    for (auto& s : g->shards) {
        s.n_live = s.n;
        if (s.n == 0 || g->ld == 0) continue;
        CU(cudaSetDevice(s.dev));
        s.buf.reset(new ShardBuf());
        s.buf->dev = s.dev;
        const int64_t cap = shard_capacity(s.n);
        CU(cudaMalloc(&s.buf->M, (size_t)cap * g->ld * 4));
        CU(cudaMalloc(&s.buf->ids, (size_t)cap * 8));
        s.buf->cap_rows = cap;
        s.M = s.buf->M; s.ids = s.buf->ids;
    }
    out = g;
    return SVSB_OK;
}

static int ensure_slabs(svsb_engine* e, int d) {
    // ~32 MB of rows per slab, 3 slabs
    int64_t rows = d > 0 ? (32ll << 20) / ((int64_t)d * 4) : 1024;
    if (rows < 16) rows = 16;
    if (rows > (1 << 20)) rows = 1 << 20;
    const int64_t bytes = rows * (int64_t)(d > 0 ? d : 1) * 4;
    if (e->slabs.size() == 3 && e->slab_bytes_rows >= bytes && e->slab_ids_cap >= rows) return SVSB_OK;
    free_slabs(e);
    e->slabs.resize(3);
    for (auto& s : e->slabs) {
        CU(cudaMallocHost(&s.rows, (size_t)bytes));
        CU(cudaMallocHost(&s.ids, (size_t)rows * 8));
        s.ev.assign(e->devs.size(), nullptr);
        s.pending.assign(e->devs.size(), 0);
        for (size_t i = 0; i < e->devs.size(); ++i) {
            CU(cudaSetDevice(e->devs[i]));
            CU(cudaEventCreateWithFlags(&s.ev[i], cudaEventDisableTiming));
        }
    }
    e->slab_bytes_rows = bytes; e->slab_ids_cap = rows;
    return SVSB_OK;
}

extern "C" int svsb_load_begin(svsb_t* e, int64_t n, int32_t d, int32_t norm_mode) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (n < 0 || d < 0) return fail(SVSB_E_INVALID, "svsb_load_begin: negative shape");
    if (norm_mode != SVSB_NORM_CHECK && norm_mode != SVSB_NORM_NORMALIZE) return fail(SVSB_E_INVALID, "svsb_load_begin: bad norm_mode");
    std::lock_guard<std::mutex> lk(e->mu);
    e->loading.reset();
    std::unique_ptr<Loading> L(new Loading());
    int rc = alloc_generation(e, n, d, L->gen);
    if (rc != SVSB_OK) return rc;
    L->norm_mode = norm_mode;
    if (n > 0 && d > 0) {
        rc = ensure_slabs(e, d);
        if (rc != SVSB_OK) return rc;
        L->slab_rows = e->slab_bytes_rows / ((int64_t)d * 4);
        if (L->slab_rows > e->slab_ids_cap) L->slab_rows = e->slab_ids_cap;
        if (L->gen->ld != d)                       // zero the padding columns once
            for (auto& s : L->gen->shards) if (s.n) {
                CU(cudaSetDevice(s.dev));
                CU(cudaMemset(s.M, 0, (size_t)s.n * L->gen->ld * 4));
                CU(cudaStreamSynchronize(cudaStreamLegacy));     // before the row copies on the (non-blocking) copy streams
            }
    }
    e->loading = std::move(L);
    return SVSB_OK;
}

static int slab_wait(svsb_engine* e, Slab& s) {
    for (size_t i = 0; i < s.pending.size(); ++i)
        if (s.pending[i]) { CU(cudaSetDevice(e->devs[i])); CU(cudaEventSynchronize(s.ev[i])); s.pending[i] = 0; }
    return SVSB_OK;
}

// copy `count` rows sitting at the start of slab `s` to their shards, asynchronously
static int slab_flush(svsb_engine* e, Loading* L, Slab& s, int64_t count) {
    Generation* g = L->gen.get();
    int64_t done = 0;
    while (done < count) {
        const int64_t grow = L->loaded + done + e->shard_row0;
        size_t si = 0;
        while (si + 1 < g->shards.size() && grow >= g->shards[si].row0 + g->shards[si].n) ++si;
        Shard& sh = g->shards[si];
        const int64_t local = grow - sh.row0;
        const int64_t take = std::min(count - done, sh.n - local);
        CU(cudaSetDevice(sh.dev));
        cudaStream_t st = e->copy_st[si];
        const float* src = s.rows + done * g->d;
        if (g->ld == g->d)
            CU(cudaMemcpyAsync(sh.M + local * g->ld, src, (size_t)take * g->d * 4, cudaMemcpyHostToDevice, st));
        else
            CU(cudaMemcpy2DAsync(sh.M + local * g->ld, (size_t)g->ld * 4, src, (size_t)g->d * 4, (size_t)g->d * 4,
                                 (size_t)take, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(sh.ids + local, s.ids + done, (size_t)take * 8, cudaMemcpyHostToDevice, st));
        CU(cudaEventRecord(s.ev[si], st));
        s.pending[si] = 1;
        done += take;
    }
    L->loaded += count;
    return SVSB_OK;
}

extern "C" int svsb_load_acquire_slab(svsb_t* e, float** rows, int64_t** emb_ids, int64_t* capacity_rows) {
    if (!e || !rows || !emb_ids || !capacity_rows) return fail(SVSB_E_INVALID, "svsb_load_acquire_slab: NULL argument");
    Loading* L = e->loading.get();
    if (!L) return fail(SVSB_E_STATE, "svsb_load_acquire_slab without svsb_load_begin");
    if (L->borrowed) return fail(SVSB_E_STATE, "a slab is already borrowed");
    if (L->slab_rows == 0) { *rows = nullptr; *emb_ids = nullptr; *capacity_rows = 0; return SVSB_OK; }
    Slab& s = e->slabs[L->cur];
    int rc = slab_wait(e, s);
    if (rc != SVSB_OK) return rc;
    *rows = s.rows; *emb_ids = s.ids;
    *capacity_rows = std::min(L->slab_rows, L->gen->n - L->loaded);
    L->borrowed = true;
    return SVSB_OK;
}

extern "C" int svsb_load_commit_slab(svsb_t* e, int64_t count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    Loading* L = e->loading.get();
    if (!L || !L->borrowed) return fail(SVSB_E_STATE, "svsb_load_commit_slab without a borrowed slab");
    L->borrowed = false;
    if (count < 0 || count > L->slab_rows) return fail(SVSB_E_INVALID, "svsb_load_commit_slab: bad count");
    if (L->loaded + count > L->gen->n) return fail(SVSB_E_STATE, "more rows supplied than announced in svsb_load_begin");
    if (count == 0) return SVSB_OK;
    int rc = slab_flush(e, L, e->slabs[L->cur], count);
    L->cur = (L->cur + 1) % (int)e->slabs.size();
    return rc;
}

extern "C" int svsb_load_rows(svsb_t* e, const float* rows, const int64_t* emb_ids, int64_t count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    Loading* L = e->loading.get();
    if (!L) return fail(SVSB_E_STATE, "svsb_load_rows without svsb_load_begin");
    if (count < 0) return fail(SVSB_E_INVALID, "svsb_load_rows: negative count");
    if (count == 0) return SVSB_OK;
    if (!emb_ids || (!rows && L->gen->d > 0)) return fail(SVSB_E_INVALID, "svsb_load_rows: NULL buffer");
    if (L->loaded + count > L->gen->n) return fail(SVSB_E_STATE, "more rows supplied than announced in svsb_load_begin");
    if (L->gen->d == 0) { L->loaded += count; return SVSB_OK; }
    const int d = L->gen->d;
    int64_t done = 0;
    while (done < count) {
        float* srows; int64_t* sids; int64_t cap;
        int rc = svsb_load_acquire_slab(e, &srows, &sids, &cap);
        if (rc != SVSB_OK) return rc;
        const int64_t take = std::min(cap, count - done);
        memcpy(srows, rows + done * d, (size_t)take * d * 4);
        memcpy(sids, emb_ids + done, (size_t)take * 8);
        rc = svsb_load_commit_slab(e, take);
        if (rc != SVSB_OK) return rc;
        done += take;
    }
    return SVSB_OK;
}

int finish_generation(svsb_engine* e, Generation* g, int norm_mode) {
    // row norms on every shard; stats reduced on the host (two words per shard)
    g->max_dev = 0.f; g->n_out_of_tol = 0;
    std::vector<u64*> stats(g->shards.size(), nullptr);
    for (size_t i = 0; i < g->shards.size(); ++i) {
        Shard& s = g->shards[i];
        if (s.n == 0 || g->ld == 0) continue;
        CU(cudaSetDevice(s.dev));
        CU(cudaMalloc(&stats[i], 16));
        CU(cudaMemsetAsync(stats[i], 0, 16, e->copy_st[i]));
        CU(launch_row_norms(e->copy_st[i], s.dev, s.M, s.n, g->d, g->ld, norm_mode == SVSB_NORM_NORMALIZE ? 1 : 0,
                            0.001f, nullptr, stats[i]));
    }
    for (size_t i = 0; i < g->shards.size(); ++i) {
        if (!stats[i]) continue;
        CU(cudaSetDevice(g->shards[i].dev));
        u64 h[2] = {0, 0};
        CU(cudaMemcpyAsync(h, stats[i], 16, cudaMemcpyDeviceToHost, e->copy_st[i]));
        CU(cudaStreamSynchronize(e->copy_st[i]));
        CU(cudaFree(stats[i]));
        const float md = bits_f32((uint32_t)h[0]);
        if (md > g->max_dev || md != md) g->max_dev = md;
        g->n_out_of_tol += (int64_t)h[1];
    }
    return SVSB_OK;
}

extern "C" int svsb_load_end(svsb_t* e, uint64_t* generation) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    Loading* L = e->loading.get();
    if (!L) return fail(SVSB_E_STATE, "svsb_load_end without svsb_load_begin");
    if (L->borrowed) { e->loading.reset(); return fail(SVSB_E_STATE, "svsb_load_end with a borrowed slab"); }
    if (L->loaded != L->gen->n) {
        char buf[160];
        snprintf(buf, sizeof buf, "svsb_load_end: %lld rows supplied, %lld announced", (long long)L->loaded, (long long)L->gen->n);
        e->loading.reset();
        return fail(SVSB_E_STATE, buf);
    }
    for (auto& s : e->slabs) { int rc = slab_wait(e, s); if (rc != SVSB_OK) { e->loading.reset(); return rc; } }
    int rc = finish_generation(e, L->gen.get(), L->norm_mode);
    if (rc != SVSB_OK) { e->loading.reset(); return rc; }
    L->gen->norm_mode = L->norm_mode;
    rc = publish_generation(e, L->gen, generation);
    e->loading.reset();
    return rc;
}

extern "C" int svsb_load_abort(svsb_t* e) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    e->loading.reset();          // frees the half-built generation (cudaFree waits for pending copies)
    for (auto& s : e->slabs) std::fill(s.pending.begin(), s.pending.end(), 0);
    return SVSB_OK;
}

extern "C" int svsb_load_synthetic(svsb_t* e, int64_t n, int32_t d, uint64_t seed, int64_t id0, int64_t id_step,
                                   uint64_t* generation) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (n < 0 || d <= 0) return fail(SVSB_E_INVALID, "svsb_load_synthetic: bad shape");
    std::shared_ptr<Generation> g;
    int rc = alloc_generation(e, n, d, g);
    if (rc != SVSB_OK) return rc;
    for (size_t i = 0; i < g->shards.size(); ++i) {
        Shard& s = g->shards[i];
        if (!s.n) continue;
        CU(cudaSetDevice(s.dev));
        CU(launch_synth(e->copy_st[i], s.dev, s.M, s.n, d, g->ld, seed, s.row0, s.ids, id0, id_step));
    }
    rc = finish_generation(e, g.get(), SVSB_NORM_NORMALIZE);
    if (rc != SVSB_OK) return rc;
    // after normalisation the deviation statistics describe the raw rows; recompute for the stored ones
    rc = finish_generation(e, g.get(), SVSB_NORM_CHECK);
    if (rc != SVSB_OK) return rc;
    return publish_generation(e, g, generation);
}

extern "C" int svsb_invalidate(svsb_t* e) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    std::shared_ptr<Generation> old;
    std::shared_ptr<Generation> pending;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        old.swap(e->current);
        pending.swap(e->pending);                    // a prepared update of the dropped generation is dropped with it
        e->has_pending = false;
    }
    return SVSB_OK;          // `old` (and its device memory) dies here unless a query still pins it
}

extern "C" int svsb_is_loaded(svsb_t* e) {
    if (!e) return 0;
    std::lock_guard<std::mutex> lk(e->mu);
    return e->current ? 1 : 0;
}

int publish_generation(svsb_engine* e, const std::shared_ptr<Generation>& g, uint64_t* generation) {
    int rc = filter_attach(e, g.get());
    if (rc != SVSB_OK) return rc;
    { std::lock_guard<std::mutex> lk(e->mu); g->id = e->next_gen++; }
    if (e->multi && (rc = multi_publish(e, g)) != SVSB_OK) return rc;   // per-device views + workspaces first
    std::lock_guard<std::mutex> lk(e->mu);
    e->current = g;
    if (generation) *generation = g->id;
    return SVSB_OK;
}

std::shared_ptr<Generation> pin(svsb_engine* e) {
    std::lock_guard<std::mutex> lk(e->mu);
    return e->current;
}

extern "C" int svsb_shape(svsb_t* e, int64_t* n, int32_t* d) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (n) *n = g->n_live;                  // what embeddings_matrix.shape[0] is to the reference: rows a query can return
    if (d) *d = g->d;
    return SVSB_OK;
}

extern "C" int svsb_norm_stats(svsb_t* e, float* max_abs_dev, int64_t* n_out_of_tolerance) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (max_abs_dev) *max_abs_dev = g->max_dev;
    if (n_out_of_tolerance) *n_out_of_tolerance = g->n_out_of_tol;
    return SVSB_OK;
}

// copy physical rows [a, b) of shard s to the host (rows: d floats each; either output may be NULL)
static int copy_rows_out(const Generation* g, const Shard& s, int64_t a, int64_t b, float* rows, int64_t* emb_ids) {
    if (a >= b) return SVSB_OK;
    CU(cudaSetDevice(s.dev));
    if (rows && g->d > 0)
        CU(cudaMemcpy2D(rows, (size_t)g->d * 4, s.M + a * g->ld, (size_t)g->ld * 4, (size_t)g->d * 4, (size_t)(b - a), cudaMemcpyDeviceToHost));
    if (emb_ids) CU(cudaMemcpy(emb_ids, s.ids + a, (size_t)(b - a) * 8, cudaMemcpyDeviceToHost));
    return SVSB_OK;
}

extern "C" int svsb_read_rows(svsb_t* e, int64_t row0, int64_t count, float* rows, int64_t* emb_ids) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (row0 < 0 || count < 0 || row0 + count > g->n_live) return fail(SVSB_E_INVALID, "svsb_read_rows: range out of bounds");
    // rows are addressed as a fresh rebuild would number them: live rows only, in row order
    int64_t logical = 0;                                         // live rows before the current position
    std::vector<uint8_t> live;
    for (auto& s : g->shards) {
        if (s.n == 0) continue;
        if (logical >= row0 + count) break;
        if (!s.live) {                                           // no tombstones in this shard: one contiguous copy
            const int64_t a = std::max(row0, logical), b = std::min(row0 + count, logical + s.n);
            if (a < b) {
                int rc = copy_rows_out(g.get(), s, a - logical, b - logical, rows ? rows + (a - row0) * g->d : nullptr,
                                       emb_ids ? emb_ids + (a - row0) : nullptr);
                if (rc != SVSB_OK) return rc;
            }
            logical += s.n;
            continue;
        }
        live.resize((size_t)s.n);
        CU(cudaSetDevice(s.dev));
        CU(cudaMemcpy(live.data(), s.live, (size_t)s.n, cudaMemcpyDeviceToHost));
        int64_t r = 0;
        while (r < s.n && logical < row0 + count) {
            if (!live[r]) { ++r; continue; }
            int64_t r1 = r;
            while (r1 < s.n && live[r1]) ++r1;                   // run of live rows [r, r1) = logical [logical, logical + r1 - r)
            const int64_t a = std::max(row0, logical), b = std::min(row0 + count, logical + (r1 - r));
            if (a < b) {
                int rc = copy_rows_out(g.get(), s, r + (a - logical), r + (b - logical), rows ? rows + (a - row0) * g->d : nullptr,
                                       emb_ids ? emb_ids + (a - row0) : nullptr);
                if (rc != SVSB_OK) return rc;
            }
            logical += r1 - r;
            r = r1;
        }
    }
    return SVSB_OK;
}

// ------------------------------------------------------------------------------------------------
// the hot path
// ------------------------------------------------------------------------------------------------
int shadow_sync(const Shard& s, int ld, int64_t fresh_from, int create, cudaStream_t st, void** out) {
    *out = nullptr;
    ShardBuf* b = s.buf.get();
    if (!b || s.n == 0 || ld == 0) return create == 2 ? fail(SVSB_E_STATE, "fp16 shadow of an empty shard") : SVSB_OK;
    const int ld16 = (ld + 7) & ~7;
    std::lock_guard<std::mutex> lk(b->m16_mu);
    CU(cudaSetDevice(s.dev));
    if (!b->M16) {
        if (create == 0) return SVSB_OK;
        const size_t bytes = (size_t)b->cap_rows * ld16 * 2;
        if (create == 1) {                               // +50 % of the matrix: only with an eighth of the device still free
            size_t fr = 0, tot = 0;
            if (cudaMemGetInfo(&fr, &tot) != cudaSuccess || fr < bytes + tot / 8) { (void)cudaGetLastError(); return SVSB_OK; }
        }
        void* p = nullptr;
        const cudaError_t ce = cudaMalloc(&p, bytes);
        if (ce != cudaSuccess) {
            (void)cudaGetLastError();
            return create == 1 ? SVSB_OK : fail(SVSB_E_NOMEM, std::string("fp16 shadow: ") + cudaGetErrorString(ce));
        }
        b->M16 = p; b->ld16 = ld16; b->m16_rows = 0;
    }
    if (fresh_from < b->m16_rows) b->m16_rows = fresh_from;
    if (b->m16_rows < s.n) {
        const int64_t r0 = b->m16_rows;
        cudaError_t ce = launch_rows_to_f16(st, s.dev, s.M + r0 * ld, s.n - r0, ld, static_cast<char*>(b->M16) + (size_t)r0 * ld16 * 2, ld16);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) { (void)cudaGetLastError(); return fail(SVSB_E_CUDA, std::string("fp16 shadow: ") + cudaGetErrorString(ce)); }
        b->m16_rows = s.n;
    }
    *out = b->M16;
    if (ld > FILTER_MAX_LD || (!b->M8 && create != 1)) return SVSB_OK;
    const int ld8 = (ld + 15) & ~15;
    if (!b->M8) {                                        // +25 % of the matrix: only with an eighth of the device still free
        // [int8 rows | f32 scales | 16-byte E word]: the int8 filter copies a partial last tile's scales in 16-byte units,
        // up to 12 bytes past scale cap_rows - 1, which the E word keeps inside this allocation (gemv8_tma_kernel)
        const size_t rows8 = (size_t)b->cap_rows * ld8, bytes = rows8 + (size_t)b->cap_rows * 4 + 16;
        size_t fr = 0, tot = 0;
        if (cudaMemGetInfo(&fr, &tot) != cudaSuccess || fr < bytes + tot / 8) { (void)cudaGetLastError(); return SVSB_OK; }
        void* p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) { (void)cudaGetLastError(); return SVSB_OK; }   // no int8 route, not an error
        float* e8 = reinterpret_cast<float*>(static_cast<char*>(p) + rows8 + (size_t)b->cap_rows * 4);
        if (cudaMemset(e8, 0, 4) != cudaSuccess) { (void)cudaGetLastError(); cudaFree(p); return SVSB_OK; }
        b->M8 = p; b->ld8 = ld8; b->m8_rows = 0;
        b->s8 = reinterpret_cast<float*>(static_cast<char*>(p) + rows8); b->e8 = e8;
    }
    if (fresh_from < b->m8_rows) b->m8_rows = fresh_from;
    if (b->m8_rows < s.n) {
        const int64_t r0 = b->m8_rows;
        cudaError_t ce = launch_rows_to_i8(st, s.dev, s.M + r0 * ld, s.n - r0, ld, static_cast<char*>(b->M8) + (size_t)r0 * ld8, ld8,
                                           b->s8 + r0, b->e8);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) { (void)cudaGetLastError(); return fail(SVSB_E_CUDA, std::string("int8 shadow: ") + cudaGetErrorString(ce)); }
        b->m8_rows = s.n;
    }
    return SVSB_OK;
}

// Single queries of a single-device engine take the int8 filter (DESIGN.md section 4, K1f8) when the view has its
// shadow: rows of norm <= 8 (fp16 range of the scaled operands), d <= FILTER_MAX_LD, and a matrix large enough to gain:
// SVSB_FILTER_MIN_MB, default 512 MB of fp32 rows.  Measured on a B200 (profiles/r05_filter_ab.txt, 1536-d rows): at
// 246 MB K1's pass is still faster than filter + threshold + re-score, at 492 MB the filter takes 25 % less time.
// shadow_sync builds the fp16 shadow here too, first, and the int8 shadow after it when that fits as well: single
// queries read only the int8 one, but the batched path (ensure_m16) and the pair search expect to find the fp16 one.
int filter_attach(svsb_engine* e, Generation* g) {
    for (auto& s : g->shards) s.M8 = nullptr;
    if (e->devs.size() != 1 || e->is_kid || g->shards.size() != 1) return SVSB_OK;
    Shard& s = g->shards[0];
    if (s.n == 0 || g->ld > FILTER_MAX_LD || !(1.0f + g->max_dev <= 8.0f)) return SVSB_OK;
    if ((double)s.n * g->ld * 4 < (double)env_int("SVSB_FILTER_MIN_MB", 512) * 1048576.0) return SVSB_OK;
    void* p = nullptr;
    int rc = shadow_sync(s, g->ld, INT64_MAX, 1, e->copy_st[0], &p);
    if (rc != SVSB_OK) return rc;
    if (p) s.M8 = s.buf->M8;
    return SVSB_OK;
}

// The route of one single query: 0 = K1, 8 = the int8 filter (DESIGN.md section 4, K1f8).  SVSB_FILTER (read per
// call): 0 forces K1; unset or any other value takes the filter wherever the view has its shadow.
// The LDG variant of K1 (SVSB_GEMV_VARIANT=1) sums in another order than the re-score, which reproduces the TMA kernel's
// bits: it turns the filter off.
static int filter_route(const Shard& s, int64_t kk) {
    if (!s.M8 || kk > K_FAST_MAX || env_int("SVSB_FILTER", 1) == 0) return 0;
    const char* v = getenv("SVSB_GEMV_VARIANT");
    if (v && atoi(v) == 1) return 0;
    return 8;
}

// The similarity pass of one query: K1, or the filter (then filter_finish before the selection).
static cudaError_t similarity_pass(cudaStream_t st, const DevWs& w, const Generation* g, const Shard& s, const float* q,
                                   int shift, int reserve_sms, int route) {
    if (route == 8)
        return launch_filter8(st, w.dev, s.M8, s.buf->s8, s.n, g->ld, s.buf->ld8, q, w.scores, w.gmax, shift, reserve_sms, s.live);
    return launch_gemv(st, w.dev, s.M, s.n, g->d, g->ld, q, w.scores, w.gmax, shift, 0, 0, 0, reserve_sms, s.live);
}
// Threshold + exact re-score: afterwards scores / gmax give launch_select K1's top-kk.
static cudaError_t filter_finish(cudaStream_t st, const DevWs& w, const Generation* g, const Shard& s, const float* q,
                                 int shift, int64_t kk) {
    return launch_filter_refine(st, w.dev, s.M, s.n, g->ld, q, w.scores, w.gmax, shift, (int)kk, (1.0f + g->max_dev) * 1.000001f,
                                s.buf->e8, s.live, w.fstate);
}

int similarity_phase(cudaStream_t st, DevWs& w, const Generation* g, const Shard& s, const float* q, int route,
                     int reserve_sms, bool pdl, cudaEvent_t* t) {
    if (t) CU(cudaEventRecord(t[0], st));
    w.gmax_dirty = true;
    {
        PdlScope scope(pdl);
        CU(similarity_pass(st, w, g, s, q, group_shift_for(s.n), reserve_sms, route));
    }
    if (t) CU(cudaEventRecord(t[1], st));
    return SVSB_OK;
}

int select_phase(cudaStream_t st, DevWs& w, const Generation* g, const Shard& s, const float* q, int route, int64_t k,
                 const SelOut& o, u64* stamps, const PeerPush* push) {
    const int shift = group_shift_for(s.n);
    const int64_t kk = std::min(k, s.n_live);
    if (route) CU(filter_finish(st, w, g, s, q, shift, kk));
    if (k <= K_FAST_MAX)
        CU(launch_select(st, w.scores, s.n, w.gmax, shift, (int)kk, s.ids, s.row0, w.cand, w.cand_cap, o.keys, o.scores, o.ids,
                         o.count, stamps, push));
    else
        CU(launch_fullsort_topk(st, w.scores, s.n, w.gmax, shift, kk, s.ids, s.row0, w.sortbuf, o.keys, o.scores, o.ids, o.count));
    w.gmax_dirty = false;
    return SVSB_OK;
}

int prepare_ws(DevWs& w, const Generation* g, const Shard& s, int64_t kk) {
    int rc;
    if ((rc = w.ensure_query(s.n, std::max<int64_t>(kk, 128), kk)) != SVSB_OK) return rc;
    return w.ensure_q(g->ld);
}

DevWs& shard_slot(svsb_engine* e, size_t i) {
    if (e->shard_ws.size() <= i) e->shard_ws.resize(i + 1);
    if (!e->shard_ws[i]) { e->shard_ws[i].reset(new DevWs()); e->shard_ws[i]->dev = e->devs[0]; }
    return *e->shard_ws[i];
}

// Argument checks shared by the synchronous and the submit / wait forms.  Returns 1 when there is nothing to compute
// (k <= 0), 0 to go on (kk set), or a negative error code.
static int query_check(const std::shared_ptr<Generation>& g, const float* q, int32_t d, int32_t k, float* out_scores,
                       int64_t* out_emb_ids, int32_t* out_count, int64_t& kk) {
    if (!out_count) return fail(SVSB_E_INVALID, "svsb_query: out_count is NULL");
    *out_count = 0;
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident (call svsb_load_* first)");
    if (g->n_live == 0 || d != g->d) {
        char buf[200];
        snprintf(buf, sizeof buf, "shapes (%lld,%d) and (%d,) not aligned: %d (dim 1) != %d (dim 0)",
                 (long long)g->n_live, g->n_live == 0 ? 0 : g->d, d, g->n_live == 0 ? 0 : g->d, d);
        return fail(SVSB_E_SHAPE, buf);
    }
    if (k <= 0) return 1;                                         // util.py:200-201
    if (!q || !out_scores || !out_emb_ids) return fail(SVSB_E_INVALID, "svsb_query: NULL buffer");
    kk = std::min<int64_t>(k, g->n_live);                        // util.py:198-199
    return 0;
}

// Single device: enqueue one query on context c.  k <= 2048: no copy-engine operation at all -- a small kernel reads
// the query from the pinned staging buffer and the selection kernel writes (score, id, count) straight into pinned host
// memory (both are device-accessible under unified addressing), so a call is 3 launches + 1 synchronize.
// reserve_sm: leave one SM to the selection kernels of OTHER in-flight queries (svsb_query_submit keeps several going).
static int enqueue_single(QueryCtx* c, const Generation* g, const float* q, int32_t d, int64_t kk, bool reserve_sm,
                          svsb_engine* chain = nullptr) {
    const Shard& s = g->shards[0];
    DevWs& w = c->ws[0];
    int rc;
    if ((rc = ctx_ensure_host(c, g->ld, kk)) != SVSB_OK) return rc;
    if ((rc = prepare_ws(w, g, s, kk)) != SVSB_OK) return rc;
    stage_queries(c->h_q, q, 1, d, g->ld);
    CU(cudaSetDevice(w.dev));
    *c->h_count = -1;
    if (kk <= K_FAST_MAX) {
        cudaStream_t gst = w.st;                                 // stream of the staging + similarity kernels
        std::unique_lock<std::mutex> chain_lk;
        if (chain) {
            chain_lk = std::unique_lock<std::mutex>(chain->chain_mu);
            if (!chain->submit_st) CU(cudaStreamCreateWithFlags(&chain->submit_st, cudaStreamNonBlocking));
            if (!c->ev_gemv) CU(cudaEventCreateWithFlags(&c->ev_gemv, cudaEventDisableTiming));
            gst = chain->submit_st;
        }
        CU(launch_stage_query(gst, c->h_q, w.d_q, g->ld));
        const int route = filter_route(s, kk);
        // programmatic dependent launch: the similarity kernel streams its first tiles under the staging kernel
        if ((rc = similarity_phase(gst, w, g, s, w.d_q, route, reserve_sm ? 1 : 0, env_int("SVSB_PDL", 1) != 0)) != SVSB_OK) return rc;
        if (chain) {
            CU(cudaEventRecord(c->ev_gemv, gst));
            chain_lk.unlock();
            CU(cudaStreamWaitEvent(w.st, c->ev_gemv, 0));
        }
        return select_phase(w.st, w, g, s, w.d_q, route, kk, {w.out_keys, c->h_scores, c->h_ids, c->h_count});
    }
    CU(cudaMemcpyAsync(w.d_q, c->h_q, (size_t)g->ld * 4, cudaMemcpyHostToDevice, w.st));
    if ((rc = similarity_phase(w.st, w, g, s, w.d_q, 0)) != SVSB_OK) return rc;
    if ((rc = select_phase(w.st, w, g, s, w.d_q, 0, kk, w.out())) != SVSB_OK) return rc;
    CU(cudaMemcpyAsync(c->h_scores, w.out_scores, (size_t)kk * 4, cudaMemcpyDeviceToHost, w.st));
    CU(cudaMemcpyAsync(c->h_ids, w.out_ids, (size_t)kk * 8, cudaMemcpyDeviceToHost, w.st));
    CU(cudaMemcpyAsync(c->h_count, w.out_count, 4, cudaMemcpyDeviceToHost, w.st));
    return SVSB_OK;
}

static int finish_single(QueryCtx* c, int64_t kk, float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    DevWs& w = c->ws[0];
    CU(cudaSetDevice(w.dev));
    CU(cudaStreamSynchronize(w.st));
    const int32_t cnt = *c->h_count;
    if (cnt != (int32_t)kk) {
        char buf[120]; snprintf(buf, sizeof buf, "internal: selection returned %d results, expected %lld", cnt, (long long)kk);
        return fail(SVSB_E_CUDA, buf);
    }
    memcpy(out_scores, c->h_scores, (size_t)kk * 4);
    memcpy(out_emb_ids, c->h_ids, (size_t)kk * 8);
    *out_count = cnt;
    return SVSB_OK;
}

static int query_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int32_t k,
                     float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    int64_t kk = 0;
    int rc = query_check(g, q, d, k, out_scores, out_emb_ids, out_count, kk);
    if (rc != 0) return rc < 0 ? rc : SVSB_OK;
    if (e->multi) return multi_query(e, g, q, d, kk, out_scores, out_emb_ids, out_count);
    CtxLease lease(e);
    if ((rc = ctx_acquire(e, lease.c)) != SVSB_OK) return rc;
    if ((rc = enqueue_single(lease.c.get(), g.get(), q, d, kk, false)) != SVSB_OK) return rc;
    return finish_single(lease.c.get(), kk, out_scores, out_emb_ids, out_count);
}

extern "C" int svsb_query(svsb_t* e, const float* q, int32_t d, int32_t k,
                          float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    return query_gen(e, pin(e), q, d, k, out_scores, out_emb_ids, out_count);
}

// ---- submit / wait: the same query with several in flight from one host thread ---------------------------------
// A pending query owns a context (its stream, workspace and pinned staging) or, on a multi-device engine, a ticket.
struct svsb_pending {
    std::unique_ptr<QueryCtx> ctx;
    svsb_ticket* ticket = nullptr;
    std::shared_ptr<Generation> gen;
    int64_t kk = 0;
};

extern "C" int svsb_query_submit(svsb_t* e, const float* q, int32_t d, int32_t k, svsb_pending_t** out) {
    if (!e || !out) return fail(SVSB_E_INVALID, "svsb_query_submit: NULL argument");
    *out = nullptr;
    auto g = pin(e);
    int32_t dummy = 0;
    float fs; int64_t fi;                                        // outputs are checked at wait time; satisfy the NULL test here
    int64_t kk = 0;
    int rc = query_check(g, q, d, k, &fs, &fi, &dummy, kk);
    if (rc < 0) return rc;
    std::unique_ptr<svsb_pending> p(new svsb_pending());
    p->gen = g; p->kk = rc == 1 ? 0 : kk;
    if (rc == 0) {
        if (e->multi) {
            if (kk > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_query_submit: k <= 2048 on a multi-device engine (use svsb_query)");
            if ((rc = multi_submit(e, g, q, d, kk, &p->ticket)) != SVSB_OK) return rc;
        } else {
            if ((rc = ctx_acquire(e, p->ctx, env_int("SVSB_SUBMIT_TIMEOUT_MS", 5000))) != SVSB_OK) return rc;
            // several queries in flight: each similarity pass leaves one SM to the (single-CTA) selections of the others
            if ((rc = enqueue_single(p->ctx.get(), g.get(), q, d, kk, sm_count(e->devs[0]) > 8, e)) != SVSB_OK) { ctx_release(e, p->ctx); return rc; }
        }
    }
    *out = p.release();
    return SVSB_OK;
}

extern "C" int svsb_query_wait(svsb_t* e, svsb_pending_t* p, float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    if (!e || !p) return fail(SVSB_E_INVALID, "svsb_query_wait: NULL argument");
    std::unique_ptr<svsb_pending> own(p);
    int rc = SVSB_OK;
    if (out_count) *out_count = 0;
    const bool bad_out = !out_count || (p->kk > 0 && (!out_scores || !out_emb_ids));
    if (p->ticket) {
        float* s = out_scores; int64_t* i = out_emb_ids; int32_t cnt = 0;
        std::vector<float> ts; std::vector<int64_t> ti;
        if (bad_out) { ts.resize((size_t)p->kk); ti.resize((size_t)p->kk); s = ts.data(); i = ti.data(); }
        rc = multi_wait(e, p->ticket, s, i, bad_out ? &cnt : out_count);      // always releases the ticket
    } else if (p->ctx) {
        if (!bad_out) rc = finish_single(p->ctx.get(), p->kk, out_scores, out_emb_ids, out_count);
        else { cudaSetDevice(p->ctx->ws[0].dev); cudaStreamSynchronize(p->ctx->ws[0].st); }
        ctx_release(e, p->ctx);
    }
    if (rc == SVSB_OK && bad_out) return fail(SVSB_E_INVALID, "svsb_query_wait: NULL buffer");
    return rc;
}

// ---- snapshots: a query handle that keeps "the arrays it fetched" alive across an invalidate ----

extern "C" int svsb_snapshot_acquire(svsb_t* e, svsb_snap_t** out) {
    if (!e || !out) return fail(SVSB_E_INVALID, "svsb_snapshot_acquire: NULL argument");
    *out = nullptr;
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    *out = new svsb_snapshot{g};
    return SVSB_OK;
}
extern "C" void svsb_snapshot_release(svsb_snap_t* s) { delete s; }
extern "C" int svsb_snapshot_shape(svsb_snap_t* s, int64_t* n, int32_t* d, uint64_t* generation) {
    if (!s || !s->gen) return fail(SVSB_E_INVALID, "snapshot is NULL");
    if (n) *n = s->gen->n_live;
    if (d) *d = s->gen->d;
    if (generation) *generation = s->gen->id;
    return SVSB_OK;
}
extern "C" int svsb_snapshot_query(svsb_t* e, svsb_snap_t* s, const float* q, int32_t d, int32_t k,
                                   float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    if (!e || !s) return fail(SVSB_E_INVALID, "svsb_snapshot_query: NULL argument");
    return query_gen(e, s->gen, q, d, k, out_scores, out_emb_ids, out_count);
}

// ------------------------------------------------------------------------------------------------
// batched queries: coarse tensor-core contraction + exact refine (coarse.cu, batch.cu; DESIGN.md section 6)
// ------------------------------------------------------------------------------------------------

struct BatchPlan {
    int64_t n = 0; int d = 0, ld = 0, ld16 = 0, kk = 0, k = 0;
    int n_tiles = 0, s_tiles = 0, tile_stride = 1; int64_t sample_rows = 0;
    int64_t sample_alloc_rows = 0;    // sample buffer rows to allocate (covers both threshold modes)
    int sample_rank = 0;              // which order statistic of the sample the filter threshold is (kk = guaranteed)
    int cand_cap = 0;
    float eps_coef = 0.f, max_row_norm = 1.f;
};

// b queries padded to whole query tiles of the coarse pass
static inline int batch_pad(int b) { return (b + COARSE_TILE_QUERIES - 1) / COARSE_TILE_QUERIES * COARSE_TILE_QUERIES; }

// Can this generation / k take the coarse path at all?  (Purely a performance gate: both paths return the same bits.)
// guaranteed: thresholds are a proven bound (the kk-th largest of the sample); else an order statistic of the sample
// that is a bound except with probability ~1e-9 per query for a random sample, verified per query by the refine
// kernel (flag 16 -> the caller redoes the batch with guaranteed thresholds).
static bool batch_plan(svsb_engine* e, const Generation* g, int32_t k, BatchPlan& P, bool guaranteed = false) {
    if (e->devs.size() != 1 || g->shards.size() != 1) return false;
    if (g->has_tombstones()) return false;     // a tombstoned row could stand in for a live one among the coarse candidates
    const Shard& s = g->shards[0];
    if (s.n != g->n || g->n < env_int("SVSB_BATCH_MIN_ROWS", 4096) || g->n > 0x7fffff00ll || g->d < 16) return false;
    const int64_t kk = std::min<int64_t>(k, g->n);
    if (kk < 1 || kk > 1024) return false;
    const float R = 1.0f + g->max_dev;
    if (!(R <= 8.0f)) return false;                               // huge / non-finite rows: fp16 operands are not safe
    P.n = g->n; P.d = g->d; P.ld = g->ld; P.ld16 = (g->d + 7) & ~7; P.kk = (int)kk; P.k = k;
    P.n_tiles = (int)((g->n + COARSE_TILE_ROWS - 1) / COARSE_TILE_ROWS);
    P.cand_cap = env_int("SVSB_BATCH_CAND_CAP", 32768);
    // sample size: the proven-bound filter lets through roughly n * kk / sample_rows candidates per query (more once
    // the 2 eps margin is subtracted); keep the expectation below cap / 4.  Statistical thresholds (below) pass about
    // n * rank / sample_rows with rank ~ 6..10 for small samples, so far fewer sampled rows do: 80 * kk measured best
    // at 1M x 768, k = 100 (profiles/r01_c3_threshold_modes.md).
    const bool stat = !guaranteed && !g->batch_guaranteed.load(std::memory_order_relaxed) && env_int("SVSB_BATCH_GUARANTEED", 0) == 0;
    auto tiles_for = [&](int64_t want) {
        int64_t st = (want + COARSE_TILE_ROWS - 1) / COARSE_TILE_ROWS;
        st = std::max<int64_t>(st, 32);
        return std::min<int64_t>(st, P.n_tiles);
    };
    const int64_t want_proven = std::max<int64_t>(320 * kk, (int64_t)(4.0 * (double)g->n * (double)kk / (double)P.cand_cap) + 1);
    int64_t want = stat ? std::max<int64_t>(80 * kk, (int64_t)(4.0 * (double)g->n * 8.0 / (double)P.cand_cap) + 1) : want_proven;
    if (const char* v = getenv("SVSB_BATCH_SAMPLE_ROWS")) want = atoll(v);
    P.s_tiles = (int)tiles_for(want);
    P.tile_stride = std::max(1, P.n_tiles / P.s_tiles);
    P.sample_rows = (int64_t)P.s_tiles * COARSE_TILE_ROWS;
    // buffers are sized for whichever mode needs more, so a chunk can be redone in the other mode in place
    P.sample_alloc_rows = std::max(P.sample_rows, tiles_for(want_proven) * COARSE_TILE_ROWS);
    P.sample_rank = (int)kk;
    if (stat) {
        // X = how many of the overall top kk fall into the sample ~ Binomial(kk, f) <= Poisson-like tail;
        // the threshold fails only if X >= rank.  rank = mean + 6 sigma + 4 puts that near 1e-9.
        const double f = std::min(1.0, (double)P.sample_rows / (double)g->n);
        const double lam = (double)kk * f;
        const int64_t r = (int64_t)std::ceil(lam + 6.0 * std::sqrt(lam) + 4.0);
        P.sample_rank = (int)std::max<int64_t>(1, std::min<int64_t>(kk, r));
    }
    // |coarse - exact| <= eps_coef * ||q|| * max||row|| + 1e-8: two fp16 roundings per product (2u + u^2, u = 2^-11),
    // fp32 accumulation inside the tensor core (d * 2^-22, generous) and the exact kernel's own rounding (d * 2^-23)
    P.eps_coef = coarse_eps_coef(g->d);
    P.max_row_norm = R * 1.000001f;
    return true;
}

static int batch_ws_get(svsb_engine* e, BatchWs*& out) {
    if (!e->batch_ws) {
        std::unique_ptr<BatchWs> w(new BatchWs());
        w->dev = e->devs[0];
        CU(cudaSetDevice(w->dev));
        CU(cudaStreamCreateWithFlags(&w->st, cudaStreamNonBlocking));
        for (auto& ev : w->ev) CU(cudaEventCreate(&ev));
        e->batch_ws = std::move(w);
    }
    out = e->batch_ws.get();
    return SVSB_OK;
}

static int batch_ws_ensure(BatchWs* w, const BatchPlan& P, int b_pad) {
    CU(cudaSetDevice(w->dev));
    const int64_t need_sample = std::max(P.sample_rows, P.sample_alloc_rows);
    if (b_pad > w->cap_b || P.ld > w->cap_ld || P.k > w->cap_k || need_sample > w->cap_sample || P.cand_cap != w->cand_cap) {
        // the sharded entry points run this workspace's kernels on the CALLER's stream: wait for the device, not for w->st only
        CU(cudaDeviceSynchronize());
        const int nb = std::max(b_pad, w->cap_b), nld = std::max(P.ld, w->cap_ld), nk = std::max(P.k, w->cap_k);
        const int64_t ns = std::max(need_sample, w->cap_sample);
        w->release_device();
        const int ld16 = (nld + 7) & ~7;
        CU(cudaMalloc(&w->dQ, (size_t)nb * nld * 4));
        CU(cudaMalloc(&w->dQ16, (size_t)nb * ld16 * 2));
        CU(cudaMalloc(&w->eps, (size_t)nb * 4)); CU(cudaMalloc(&w->thr, (size_t)nb * 4));
        CU(cudaMalloc(&w->flags, (size_t)nb * 4)); CU(cudaMalloc(&w->cand_cnt, (size_t)nb * 4)); CU(cudaMalloc(&w->stats, (size_t)nb * 4));
        CU(cudaMalloc(&w->sample, (size_t)nb * ns * 4));
        CU(cudaMalloc(&w->cand, (size_t)nb * P.cand_cap * 8));
        CU(cudaMalloc(&w->rs.rows, (size_t)nb * REFINE_SURVIVOR_CAP * 4)); CU(cudaMalloc(&w->rs.keys, (size_t)nb * REFINE_SURVIVOR_CAP * 8));
        CU(cudaMalloc(&w->rs.cnt, (size_t)nb * 4)); CU(cudaMalloc(&w->rs.ver, (size_t)nb * 4));
        CU(cudaMalloc(&w->tops, (size_t)nb * SAMPLE_TOPX * 4));
        CU(cudaMalloc(&w->o_scores, (size_t)nb * nk * 4)); CU(cudaMalloc(&w->o_ids, (size_t)nb * nk * 8)); CU(cudaMalloc(&w->o_counts, (size_t)nb * 4));
        CU(cudaMallocHost(&w->h_Q, (size_t)nb * nld * 4));
        CU(cudaMallocHost(&w->h_scores, (size_t)nb * nk * 4)); CU(cudaMallocHost(&w->h_ids, (size_t)nb * nk * 8));
        CU(cudaMallocHost(&w->h_counts, (size_t)nb * 4)); CU(cudaMallocHost(&w->h_flags, (size_t)nb * 4));
        CU(cudaMallocHost(&w->h_stats, (size_t)nb * 4)); CU(cudaMallocHost(&w->h_cnt, (size_t)nb * 4));
        w->cap_b = nb; w->cap_ld = nld; w->cap_k = nk; w->cap_sample = ns; w->cand_cap = P.cand_cap;
    }
    return SVSB_OK;
}

// fp16 shadow of the matrix: the shard buffer's (shared by the generations of one lineage), covering this view's rows
static int ensure_m16(Generation* g, const BatchPlan& P, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g->m16_mu);
    if (g->M16) return SVSB_OK;
    void* p = nullptr;
    int rc = shadow_sync(g->shards[0], g->ld, INT64_MAX, 2, st, &p);
    if (rc != SVSB_OK) return rc;
    g->M16 = p; g->ld16 = P.ld16;
    return SVSB_OK;
}

// The batch workspace, sized for b queries of plan P, over the generation's fp16 shadow (converted on st, the stream the
// batch's kernels run on; null: the workspace's own).  The caller holds batch_mu.
static int batch_acquire(svsb_engine* e, Generation* g, const BatchPlan& P, int b, cudaStream_t st, BatchWs*& w) {
    int rc = batch_ws_get(e, w);
    if (rc != SVSB_OK) return rc;
    if ((rc = ensure_m16(g, P, st ? st : w->st)) != SVSB_OK) return rc;
    return batch_ws_ensure(w, P, batch_pad(b));
}

// The two phases of the pipeline for b (<= COARSE_MAX_BATCH) device-resident fp32 queries dQ[b][ld], enqueued on st
// (the workspace's own stream, or the caller's in the sharded path).  Between them a threshold kernel fills w->thr.
// Sample phase: the queries -> fp16 (with their error bounds, flags and candidate counts reset), then the sample pass.
static int batch_sample(BatchWs* w, const Generation* g, const BatchPlan& P, const float* dQ, int b, cudaStream_t st) {
    const int b_pad = batch_pad(b);
    CU(cudaSetDevice(w->dev));
    CU(launch_queries_to_f16(st, dQ, b, b_pad, P.d, P.ld, w->dQ16, P.ld16, P.eps_coef, P.max_row_norm, w->eps, w->thr, w->flags, w->cand_cnt));
    CU(launch_coarse_gemm(st, w->dev, 1, g->M16, P.n, w->dQ16, b_pad, P.ld16, P.s_tiles, P.tile_stride,
                          nullptr, nullptr, nullptr, 0, w->sample, P.sample_rows));
    return SVSB_OK;
}

// Filter + refine phase: the filter pass keeps every row whose coarse score reaches w->thr, the refine re-scores them
// exactly into `out` (mode: REFINE_* flags; push: records into the peers' windows).  w->flags[q] != 0: query q needs
// the exact path.  time_coarse: bracket the filter pass with w->ev[2], w->ev[3].
static int batch_filter_refine(BatchWs* w, const Generation* g, const BatchPlan& P, const float* dQ, int b, cudaStream_t st,
                               const RefineOut& out, int mode = 0, const BatchPush* push = nullptr, bool time_coarse = false) {
    const Shard& s = g->shards[0];
    if (time_coarse) CU(cudaEventRecord(w->ev[2], st));
    CU(launch_coarse_gemm(st, w->dev, 0, g->M16, P.n, w->dQ16, batch_pad(b), P.ld16, P.n_tiles, 1,
                          w->thr, w->cand, w->cand_cnt, P.cand_cap, nullptr, 0));
    if (time_coarse) CU(cudaEventRecord(w->ev[3], st));
    CU(launch_refine(st, s.M, P.n, P.ld, s.ids, s.row0, dQ, b, P.ld, P.k, w->cand, w->cand_cnt, P.cand_cap, w->eps, w->thr, w->flags,
                     out, w->stats, &w->rs, mode, push));
    return SVSB_OK;
}

// The whole pipeline with this shard's own thresholds.  out == nullptr: results go to w->o_scores / o_ids [b][k],
// w->o_counts[b].
static int batch_enqueue(BatchWs* w, const Generation* g, const BatchPlan& P, const float* dQ, int b, bool time_coarse,
                         cudaStream_t st, const RefineOut* out = nullptr) {
    int rc = batch_sample(w, g, P, dQ, b, st);
    if (rc != SVSB_OK) return rc;
    CU(launch_sample_threshold(st, w->sample, P.sample_rows, b, P.sample_rank, w->eps, w->thr));
    if (env_int("SVSB_DEBUG_NO_SURVIVORS", 0)) {          // measurement aid: thresholds +inf -> the filter pass keeps nothing
        std::vector<uint32_t> inf((size_t)batch_pad(b), 0x7f800000u);
        CU(cudaMemcpyAsync(w->thr, inf.data(), inf.size() * 4, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
    }
    const RefineOut own{w->o_scores, nullptr, w->o_ids, (int64_t)P.k, w->o_counts, 1};
    return batch_filter_refine(w, g, P, dQ, b, st, out ? *out : own, 0, nullptr, time_coarse);
}

// Did enough statistical thresholds fail verification (flag 16) that the chunk should be redone with guaranteed ones?
// A handful of failures is cheaper to hand to the single-query kernels; many mean the sample is not representative
// (rows stored in an order correlated with the queries), so the generation switches modes for good.
static bool batch_thresholds_failed(Generation* g, const BatchPlan& P, const int32_t* h_flags, int b) {
    if (P.sample_rank >= P.kk) return false;
    int bad = 0;
    for (int i = 0; i < b; ++i) bad += (h_flags[i] & (REFINE_FLAG_THRESHOLD_HIGH | 4)) ? 1 : 0;   // 4 = fewer than kk candidates: threshold far too high
    if (bad <= std::max(2, b / 256)) return false;
    g->batch_guaranteed.store(true, std::memory_order_relaxed);
    return true;
}

// Run bc device-resident queries dQ[bc][ld] (one chunk of at most COARSE_MAX_BATCH) through the pipeline on st and bring
// their flags to w->h_flags, with ONE synchronisation of st: fetch() enqueues the caller's result copies before it.
// If too many statistical thresholds failed, P is re-planned with guaranteed ones and the chunk redone in place.
template <class Fetch>
static int batch_run_chunk(svsb_engine* e, Generation* g, BatchPlan& P, BatchWs* w, cudaStream_t st, const float* dQ, int bc,
                           const RefineOut* out, Fetch fetch) {
    for (int attempt = 0; attempt < 2; ++attempt) {
        int rc = batch_enqueue(w, g, P, dQ, bc, false, st, out);
        if (rc != SVSB_OK || (rc = fetch()) != SVSB_OK) return rc;
        CU(cudaMemcpyAsync(w->h_flags, w->flags, (size_t)bc * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (!batch_thresholds_failed(g, P, w->h_flags, bc)) break;
        batch_plan(e, g, P.k, P, true);
    }
    return SVSB_OK;
}

static bool is_pinned_host(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost;
}

extern "C" int svsb_host_alloc(size_t bytes, void** out) {
    if (!out) return fail(SVSB_E_INVALID, "svsb_host_alloc: NULL argument");
    *out = nullptr;
    if (bytes == 0) bytes = 1;
    cudaError_t ce = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    if (ce != cudaSuccess) { (void)cudaGetLastError(); return fail(ce == cudaErrorMemoryAllocation ? SVSB_E_NOMEM : SVSB_E_CUDA, std::string("svsb_host_alloc: ") + cudaGetErrorString(ce)); }
    return SVSB_OK;
}
extern "C" int svsb_host_free(void* p) {
    if (p) CU(cudaFreeHost(p));
    return SVSB_OK;
}

// ---- small exact batches: ONE pass over the matrix for up to 8 warps' worth of queries (gemv.cu: gemv_tma_mq_kernel),
//      then one selection CTA per query.  Same bits as the single-query kernels; no fp16 shadow, any k <= 2048, tombstones ok.
struct MqPlan { int bq = 0, chunk = 0, max_b = 0; };
static bool mq_plan(const Generation* g, int64_t kk, MqPlan& P) {
    if (env_int("SVSB_MQ", 1) == 0 || g->shards.size() != 1 || g->n_live == 0) return false;
    P.bq = gemv_mq_queries_per_warp(g->ld);
    if (P.bq == 0 || kk < 1 || kk > K_FAST_MAX) return false;
    // per launch: `groups` x bq queries, each streamed byte read `groups` times from shared memory.  4 groups is the
    // measured sweet spot (profiles/r02_mq_sweep.txt); bounded by 2 GB of score vectors.
    P.chunk = std::min(8, std::max(1, env_int("SVSB_MQ_GROUPS", 4))) * P.bq;
    const int64_t by_mem = std::max<int64_t>(1, (2ll << 30) / std::max<int64_t>(g->shards[0].n * 4, 1));
    if (P.chunk > by_mem) P.chunk = (int)by_mem;
    // Which path answers a batch when the tensor-core coarse pass is ALSO available (profiles/r02_mq_sweep.txt, 1M rows):
    // the coarse pass reads the fp16 shadow (half the bytes) and costs ~0.72 ms at d = 1536 / 0.40 ms at d = 768 for any
    // b <= 256 while k is small, so it wins from 4 queries on (multi-query: 0.96 ms for 4, 1.2 ms for 8); its exact refine
    // grows with k, and at k = 1000 (d = 3072) it needs 8.3 ms for 4 queries against 1.8 ms here -- large k stays exact
    // multi-query at every batch size.  Batches the coarse pass cannot take (tombstones, k > 1024, no room for the
    // shadow matrix) run as multi-query passes regardless.
    P.max_b = env_int("SVSB_MQ_MAX", kk > 256 ? 0x7fffffff : 3);
    return P.chunk >= 2;
}

static int mq_ws_get(svsb_engine* e, MqWs*& out) {
    if (!e->mq_ws) { e->mq_ws.reset(new MqWs()); e->mq_ws->dev = e->devs[0]; }
    out = e->mq_ws.get();
    return SVSB_OK;
}

// Multi-query passes over b queries, P.chunk at a time: each query's top-kk list goes to the records `recs` or, with
// recs.base null, to the workspace's dense [chunk][kk] outputs.  Per chunk the workspace is sized and its own stream
// drained (its zeroing is done, its staging buffer free), stage(w, c0, bc, dQ) points dQ at the chunk's device-resident
// queries [bc][ld], gemv + selection run on st (null: the workspace's stream) and drain(w, c0, bc) takes the results.
// The caller holds batch_mu.
template <class Stage, class Drain>
static int mq_run(svsb_engine* e, const Generation* g, const MqPlan& P, int32_t b, int64_t kk, cudaStream_t st, const RecordView& recs,
                  Stage stage, Drain drain) {
    MqWs* w = nullptr;
    int rc = mq_ws_get(e, w);
    if (rc != SVSB_OK) return rc;
    const Shard& s = g->shards[0];
    for (int32_t c0 = 0; c0 < b; c0 += P.chunk) {
        const int bc = std::min<int32_t>(P.chunk, b - c0);
        if ((rc = w->ensure(std::min<int32_t>(P.chunk, b), s.n, g->ld, kk)) != SVSB_OK) return rc;
        CU(cudaStreamSynchronize(w->st));
        const float* dQ = nullptr;
        if ((rc = stage(w, c0, bc, dQ)) != SVSB_OK) return rc;
        cudaStream_t run = st ? st : w->st;
        SelectStrides ss; ss.keys = kk; ss.oscores = kk; ss.ids = kk; ss.count = 1;
        u64* keys = w->o_keys; int64_t* ids = w->o_ids; int32_t* counts = w->o_counts;
        if (recs.base) { ss = recs.select_strides(kk); keys = recs.keys(c0); ids = recs.ids(c0); counts = recs.count(c0); }
        ss.scores = w->cap_n; ss.gmax = w->G; ss.cand = w->cand_cap;
        const int shift = group_shift_for(w->cap_n);             // group layout of the workspace (>= this shard's rows)
        CU(cudaSetDevice(w->dev));
        w->gmax_dirty = true;
        CU(launch_gemv_mq(run, w->dev, s.M, s.n, g->d, g->ld, dQ, bc, w->scores, w->cap_n, w->gmax, w->G, shift, s.live, 0));
        CU(launch_select_batch(run, bc, ss, w->scores, s.n, w->gmax, shift, (int)std::min<int64_t>(kk, s.n_live), s.ids, s.row0, w->cand,
                               w->cand_cap, keys, w->o_scores, ids, counts));
        w->gmax_dirty = false;
        if ((rc = drain(w, c0, bc)) != SVSB_OK) return rc;
    }
    return SVSB_OK;
}

static int query_batch_mq(svsb_engine* e, const std::shared_ptr<Generation>& g, const MqPlan& P, const float* Q, int32_t b, int32_t d,
                          int32_t k, int64_t kk, float* out_scores, int64_t* out_emb_ids, int32_t* out_counts) {
    std::lock_guard<std::mutex> lk(e->batch_mu);
    const int ld = g->ld;
    auto stage = [&](MqWs* w, int c0, int bc, const float*& dQ) -> int {
        stage_queries(w->h_Q, Q + (size_t)c0 * d, bc, d, ld);
        CU(cudaMemcpyAsync(w->dQ, w->h_Q, (size_t)bc * ld * 4, cudaMemcpyHostToDevice, w->st));
        dQ = w->dQ;
        return SVSB_OK;
    };
    auto drain = [&](MqWs* w, int c0, int bc) -> int {
        CU(cudaMemcpy2DAsync(out_scores + (int64_t)c0 * k, (size_t)k * 4, w->o_scores, (size_t)kk * 4, (size_t)kk * 4, (size_t)bc, cudaMemcpyDeviceToHost, w->st));
        CU(cudaMemcpy2DAsync(out_emb_ids + (int64_t)c0 * k, (size_t)k * 8, w->o_ids, (size_t)kk * 8, (size_t)kk * 8, (size_t)bc, cudaMemcpyDeviceToHost, w->st));
        CU(cudaMemcpyAsync(out_counts + c0, w->o_counts, (size_t)bc * 4, cudaMemcpyDeviceToHost, w->st));
        CU(cudaStreamSynchronize(w->st));
        return SVSB_OK;
    };
    return mq_run(e, g.get(), P, b, kk, nullptr, RecordView{}, stage, drain);
}

static int query_batch_loop(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* Q, int32_t b, int32_t d, int32_t k,
                            float* out_scores, int64_t* out_emb_ids, int32_t* out_counts) {
    const int64_t kstride = k > 0 ? k : 0;
    for (int32_t i = 0; i < b; ++i) {
        int rc = query_gen(e, g, Q + (int64_t)i * d, d, k, out_scores ? out_scores + i * kstride : nullptr,
                           out_emb_ids ? out_emb_ids + i * kstride : nullptr, out_counts + i);
        if (rc != SVSB_OK) return rc;
    }
    return SVSB_OK;
}

static int query_batch_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* Q, int32_t b, int32_t d, int32_t k,
                           float* out_scores, int64_t* out_emb_ids, int32_t* out_counts) {
    if (b < 0) return fail(SVSB_E_INVALID, "svsb_query_batch: negative batch");
    if (b == 0) return SVSB_OK;
    if (!Q || !out_counts) return fail(SVSB_E_INVALID, "svsb_query_batch: NULL buffer");
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident (call svsb_load_* first)");
    for (int32_t i = 0; i < b; ++i) out_counts[i] = 0;
    BatchPlan P;
    if (e->multi && g->n_live > 0 && d == g->d && k > 0 && b >= 2 && out_scores && out_emb_ids)
        return multi_query_batch(e, g, Q, b, d, k, out_scores, out_emb_ids, out_counts);
    bool coarse = g->n_live > 0 && d == g->d && k > 0 && b >= env_int("SVSB_BATCH_MIN", 4) && batch_plan(e, g.get(), k, P);
    MqPlan MP;
    if (g->n_live > 0 && d == g->d && k > 0 && b >= 2 && out_scores && out_emb_ids && !e->multi &&
        mq_plan(g.get(), std::min<int64_t>(k, g->n_live), MP) && (b <= MP.max_b || !coarse))
        return query_batch_mq(e, g, MP, Q, b, d, k, std::min<int64_t>(k, g->n_live), out_scores, out_emb_ids, out_counts);
    if (!coarse)                                      // same results, one similarity pass per query
        return query_batch_loop(e, g, Q, b, d, k, out_scores, out_emb_ids, out_counts);
    if (!out_scores || !out_emb_ids) return fail(SVSB_E_INVALID, "svsb_query_batch: NULL buffer");

    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = nullptr;
    int rc = batch_acquire(e, g.get(), P, std::min<int32_t>(b, COARSE_MAX_BATCH), nullptr, w);
    if (rc == SVSB_E_NOMEM) return query_batch_loop(e, g, Q, b, d, k, out_scores, out_emb_ids, out_counts);
    if (rc != SVSB_OK) return rc;
    // Page-locked caller buffers (svsb_host_alloc, cudaHostRegister, torch pin_memory) are DMA'd from / into directly;
    // pageable ones are staged through the workspace's pinned buffers.
    const bool q_direct = is_pinned_host(Q) && d == P.ld;
    const bool out_direct = is_pinned_host(out_scores) && is_pinned_host(out_emb_ids);
    for (int32_t c0 = 0; c0 < b; c0 += COARSE_MAX_BATCH) {
        const int bc = std::min<int32_t>(COARSE_MAX_BATCH, b - c0);
        const float* src = Q + (size_t)c0 * d;
        if (!q_direct) {
            stage_queries(w->h_Q, src, bc, d, P.ld);
            src = w->h_Q;
        }
        float* dst_scores = out_direct ? out_scores + (int64_t)c0 * k : w->h_scores;
        int64_t* dst_ids = out_direct ? out_emb_ids + (int64_t)c0 * k : w->h_ids;
        CU(cudaSetDevice(w->dev));
        CU(cudaMemcpyAsync(w->dQ, src, (size_t)bc * P.ld * 4, cudaMemcpyHostToDevice, w->st));
        rc = batch_run_chunk(e, g.get(), P, w, w->st, w->dQ, bc, nullptr, [&]() -> int {
            CU(cudaMemcpyAsync(dst_scores, w->o_scores, (size_t)bc * k * 4, cudaMemcpyDeviceToHost, w->st));
            CU(cudaMemcpyAsync(dst_ids, w->o_ids, (size_t)bc * k * 8, cudaMemcpyDeviceToHost, w->st));
            CU(cudaMemcpyAsync(w->h_counts, w->o_counts, (size_t)bc * 4, cudaMemcpyDeviceToHost, w->st));
            return SVSB_OK;
        });
        if (rc != SVSB_OK) return rc;
        for (int i = 0; i < bc; ++i) {
            const int64_t o = (int64_t)(c0 + i) * k;
            if (w->h_flags[i] == 0 && w->h_counts[i] == P.kk) {
                if (!out_direct) {
                    memcpy(out_scores + o, w->h_scores + (size_t)i * k, (size_t)P.kk * 4);
                    memcpy(out_emb_ids + o, w->h_ids + (size_t)i * k, (size_t)P.kk * 8);
                }
                out_counts[c0 + i] = P.kk;
            } else {                                   // overflowed / untrusted query: exact single-query kernels
                rc = query_gen(e, g, Q + (size_t)(c0 + i) * d, d, k, out_scores + o, out_emb_ids + o, out_counts + c0 + i);
                if (rc != SVSB_OK) return rc;
            }
        }
    }
    return SVSB_OK;
}

extern "C" int svsb_query_batch(svsb_t* e, const float* Q, int32_t b, int32_t d, int32_t k,
                                float* out_scores, int64_t* out_emb_ids, int32_t* out_counts) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    return query_batch_gen(e, pin(e), Q, b, d, k, out_scores, out_emb_ids, out_counts);
}
extern "C" int svsb_snapshot_query_batch(svsb_t* e, svsb_snap_t* s, const float* Q, int32_t b, int32_t d, int32_t k,
                                         float* out_scores, int64_t* out_emb_ids, int32_t* out_counts) {
    if (!e || !s) return fail(SVSB_E_INVALID, "svsb_snapshot_query_batch: NULL argument");
    return query_batch_gen(e, s->gen, Q, b, d, k, out_scores, out_emb_ids, out_counts);
}

// ------------------------------------------------------------------------------------------------
// pairwise top pairs: document_top_pairwise_scores' compute (reference src/svs/kb.py:1642-1671, 1208-1243;
// src/svs/util.py:206-233) on the coarse tensor-core pass + exact refine (pairs.cu)
// ------------------------------------------------------------------------------------------------
// Static plan of the pass over G row shards: device a runs the upper triangle of its own shard, then the full rectangles
// (a, a + t mod G) for t = 1 .. ceil(G/2) - 1; for even G the opposite rectangle (a, a + G/2) is split in half between
// its two devices (a takes all of its rows against the first half of the other shard's, the other device its second
// half against all of a's).  Invariants:
//   1. every unordered pair of distinct global rows is covered by exactly one task of one device;
//   2. with equal shards no device gets more than 1/G of the pair work plus a few percent (the odd half row of a split).
// Empty tasks are left out.  tests/test_pairs_multi_logic.py restates this function.
std::vector<std::vector<PairTask>> pairs_plan(const std::vector<int64_t>& shard_rows) {
    const int G = (int)shard_rows.size();
    std::vector<std::vector<PairTask>> plan((size_t)G);
    auto add = [&](int dev, int peer, int64_t m0, int64_t m1, int64_t q0, int64_t q1) {
        if (m1 > m0 && q1 > q0 && (peer != dev || m1 - m0 >= 2)) plan[(size_t)dev].push_back(PairTask{peer, m0, m1, q0, q1});
    };
    for (int a = 0; a < G; ++a) {
        add(a, a, 0, shard_rows[a], 0, shard_rows[a]);
        for (int t = 1; t < (G + 1) / 2; ++t) {
            const int b = (a + t) % G;
            add(a, b, 0, shard_rows[a], 0, shard_rows[b]);
        }
    }
    if (G % 2 == 0)
        for (int a = 0; a < G / 2; ++a) {
            const int b = a + G / 2;
            const int64_t h = shard_rows[b] / 2;
            add(a, b, 0, shard_rows[a], 0, h);
            add(b, a, h, shard_rows[b], 0, shard_rows[a]);
        }
    return plan;
}

PairRows pair_rows_of(const std::vector<Generation*>& views) {
    PairRows t;
    t.n = (int)views.size();
    const int64_t base = views[0]->shards[0].row0;
    for (int s = 0; s < t.n; ++s) {
        const Shard& sh = views[s]->shards[0];
        t.row0[s] = sh.row0 - base; t.M[s] = sh.M; t.ids[s] = sh.ids;
    }
    t.row0[t.n] = t.row0[t.n - 1] + views[t.n - 1]->shards[0].n;
    return t;
}

constexpr int PAIRS_BLOCK = 1024;                  // query rows per coarse block

float pairs_eps2(int d, float R) {
    const float eps = (9.765625e-4f + 2.384185791015625e-7f + (float)d * (2.384185791015625e-7f + 1.1920928955078125e-7f))
                      * (R * 1.000001f) * (R * 1.000001f) + 1e-8f;
    return 2.0f * eps;
}

int pairs_dev_prepare(svsb_engine* e, Generation* g, int64_t n, float eps2, PairsDev& r) {
    r.g = g; r.n = n; r.eps2 = eps2;
    const int64_t N = g->shards[0].n;
    if (N == 0 || g->d == 0) return SVSB_OK;       // no rows here: nothing to compute, nothing for a peer to read
    BatchPlan P;
    P.n = N; P.d = g->d; P.ld = g->ld; P.ld16 = (g->d + 7) & ~7; P.kk = 1; P.k = 1;
    P.n_tiles = (int)((N + COARSE_TILE_ROWS - 1) / COARSE_TILE_ROWS);
    P.cand_cap = env_int("SVSB_BATCH_CAND_CAP", 32768);
    const int B = PAIRS_BLOCK;
    // bootstrap sample (only when a first block at threshold -inf would overflow the per-row lists)
    r.bootstrap = N >= 2048;
    int64_t want_rows = std::max<int64_t>(std::max<int64_t>(4096, n / 16 + 1),
                                          (int64_t)((double)N * (double)n / (64.0 * (double)P.cand_cap)) + 1);
    int64_t st_ = std::max<int64_t>((want_rows + COARSE_TILE_ROWS - 1) / COARSE_TILE_ROWS, 32);
    st_ = std::min<int64_t>(st_, P.n_tiles);
    P.s_tiles = (int)st_; P.tile_stride = std::max(1, P.n_tiles / P.s_tiles);
    P.sample_rows = (int64_t)P.s_tiles * COARSE_TILE_ROWS;
    r.ld16 = P.ld16; r.cand_cap = P.cand_cap; r.s_tiles = P.s_tiles; r.tile_stride = P.tile_stride; r.sample_rows = P.sample_rows;

    BatchWs* w = nullptr;
    int rc = batch_ws_get(e, w);
    if (rc != SVSB_OK) return rc;
    if ((rc = ensure_m16(g, P, w->st)) != SVSB_OK) return rc;
    {   // the sample buffer holds 256 x sample_rows floats: size it through the (b_pad x sample_rows) allocation
        BatchPlan Pa = P;
        Pa.sample_rows = std::max<int64_t>(1, (256 * P.sample_rows + B - 1) / B);
        if ((rc = batch_ws_ensure(w, Pa, B)) != SVSB_OK) return rc;
    }
    CU(cudaSetDevice(w->dev));
    r.w = w; r.st = w->st; r.bufs.dev = w->dev;
    r.LC = std::max<int64_t>(1ll << 22, 16 * n);
    for (int i = 0; i < 2; ++i) { CU(r.bufs.get(&r.lo[i], (size_t)r.LC)); CU(r.bufs.get(&r.lp[i], (size_t)r.LC)); CU(r.bufs.get(&r.lstate[i], 2)); }
    CU(r.bufs.get(&r.thr, 1));
    const uint32_t neg_inf = 0xff800000u;
    CU(cudaMemcpyAsync(r.thr, &neg_inf, 4, cudaMemcpyHostToDevice, r.st));
    CU(cudaMemsetAsync(r.lstate[0], 0, 16, r.st));
    return SVSB_OK;
}

int pairs_dev_coarse(PairsDev& r, int self, const std::vector<PairTask>& tasks, const std::vector<PairShadow>& shadows, const PairRows& rows) {
    r.C = 0;
    if (!r.w) return SVSB_OK;
    BatchWs* w = r.w;
    Generation* g = r.g;
    cudaStream_t st = r.st;
    const int64_t N = g->shards[0].n;
    const int B = PAIRS_BLOCK;
    const int n = (int)r.n;
    const size_t row16 = (size_t)r.ld16 * 2;
    const char* m16 = reinterpret_cast<const char*>(g->M16);
    CU(cudaSetDevice(w->dev));
    if (r.bootstrap) {
        CU(launch_coarse_gemm(st, w->dev, 1, g->M16, N, g->M16, 256, r.ld16, r.s_tiles, r.tile_stride, nullptr, nullptr, nullptr, 0,
                              w->sample, r.sample_rows, /*q_rows=*/std::min<int64_t>(N, 256), /*tri_q0=*/0));
        CU(launch_pairs_tau(st, nullptr, w->sample, 256 * r.sample_rows, nullptr, 0, n, r.eps2, r.thr));
    }
    // bq query rows (q16, q_rows of them readable) against m_rows matrix rows (m16op); global rows of the first of each
    auto block = [&](const char* m16op, int64_t m_rows, const void* q16, int64_t q_rows, int bq, int64_t tri_q0,
                     int64_t q_row0, int64_t m_row0) -> int {
        const int cur = r.cur;
        const int b_pad = batch_pad(bq);
        const int m_tiles = (int)((m_rows + COARSE_TILE_ROWS - 1) / COARSE_TILE_ROWS);
        CU(launch_pairs_fill_thr(st, w->thr, b_pad, bq, r.thr));
        CU(cudaMemsetAsync(w->cand_cnt, 0, (size_t)b_pad * 4, st));
        CU(launch_coarse_gemm(st, w->dev, 0, m16op, m_rows, q16, b_pad, r.ld16, m_tiles, 1, w->thr,
                              w->cand, w->cand_cnt, r.cand_cap, nullptr, 0, q_rows, tri_q0));
        CU(launch_pairs_gather(st, w->cand, w->cand_cnt, r.cand_cap, bq, q_row0, m_row0, r.lo[cur], r.lp[cur], r.LC, r.lstate[cur]));
        CU(launch_pairs_tau(st, r.lo[cur], nullptr, 0, r.lstate[cur], r.LC, n, r.eps2, r.thr));
        CU(cudaMemsetAsync(r.lstate[cur ^ 1], 0, 16, st));
        CU(launch_pairs_compact(st, w->dev, r.lo[cur], r.lp[cur], r.lstate[cur], r.LC, r.lo[cur ^ 1], r.lp[cur ^ 1], r.lstate[cur ^ 1], r.thr));
        r.cur = cur ^ 1;
        return SVSB_OK;
    };
    const int64_t row0 = rows.row0[self];
    int rc;
    for (const PairTask& t : tasks) {
        if (t.peer == self) {      // upper triangle: the shard itself plays the queries from row q0 on (coarse pairwise mode)
            for (int64_t q0 = 0; q0 + 1 < N; q0 += B)
                if ((rc = block(m16, N, m16 + (size_t)q0 * row16, N - q0, (int)std::min<int64_t>(B, N - q0), q0, row0 + q0, row0)) != SVSB_OK)
                    return rc;
        } else {                   // rectangle: blocks of the peer's fp16 rows copied next to this shard, no mask
            const PairShadow& pv = shadows[(size_t)t.peer];
            for (int64_t q0 = t.q0; q0 < t.q1; q0 += B) {
                const int bq = (int)std::min<int64_t>(B, t.q1 - q0);
                const char* src = reinterpret_cast<const char*>(pv.M16) + (size_t)q0 * row16;
                if (pv.dev >= 0) CU(cudaMemcpyPeerAsync(w->dQ16, w->dev, src, pv.dev, (size_t)bq * row16, st));
                else CU(cudaMemcpyAsync(w->dQ16, src, (size_t)bq * row16, cudaMemcpyDefault, st));
                if ((rc = block(m16 + (size_t)t.m0 * row16, t.m1 - t.m0, w->dQ16, bq, bq, -1, rows.row0[t.peer] + q0, row0 + t.m0)) != SVSB_OK)
                    return rc;
            }
        }
    }
    unsigned long long hstate[2] = {0, 0};
    CU(cudaMemcpyAsync(hstate, r.lstate[r.cur], 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (hstate[1] != 0)
        return fail(SVSB_E_NOMEM, hstate[1] & 1 ? "svsb_top_pairs: a row has more than 32768 near-tied partners (raise SVSB_BATCH_CAND_CAP)"
                                                : "svsb_top_pairs: too many near-tied pairs for the candidate list");
    r.C = (int64_t)hstate[0];
    return SVSB_OK;
}

int pairs_dev_alloc(PairsDev& r) {
    r.kl = std::min(r.n, r.C);
    if (r.kl == 0) return SVSB_OK;
    CU(cudaSetDevice(r.w->dev));
    const int64_t C = r.C, n = r.kl;
    r.np2 = next_pow2(C); if (r.np2 < 2048) r.np2 = 2048;
    r.shift = group_shift_for(C);
    const int64_t G = (C + ((int64_t)1 << r.shift) - 1) >> r.shift;
    DevBufs& b = r.bufs;
    CU(b.get(&r.keys, (size_t)r.np2)); CU(b.get(&r.scores, (size_t)C)); CU(b.get(&r.sortbuf, (size_t)r.np2));
    CU(b.get(&r.gmax, (size_t)G)); CU(b.get(&r.o_keys, (size_t)n)); CU(b.get(&r.o_scores, (size_t)n)); CU(b.get(&r.o_sel, (size_t)n));
    CU(b.get(&r.o_cnt, 16)); CU(b.get(&r.o_a, (size_t)n)); CU(b.get(&r.o_b, (size_t)n));
    return SVSB_OK;
}

int pairs_dev_finish(PairsDev& r, const PairRows& rows, const int64_t* ids) {
    if (r.kl == 0) return SVSB_OK;
    cudaStream_t st = r.st;
    CU(cudaSetDevice(r.w->dev));
    CU(launch_pairs_sortkeys(st, r.lp[r.cur], r.C, r.np2, r.keys));
    CU(launch_sort_keys_desc(st, r.keys, r.np2));                 // ascending (i, j)
    CU(launch_pairs_rescore(st, r.w->dev, rows, r.g->ld, r.keys, r.C, r.scores));
    CU(launch_fullsort_topk(st, r.scores, r.C, r.gmax, r.shift, r.kl, nullptr, 0, r.sortbuf, r.o_keys, r.o_scores, r.o_sel, r.o_cnt));
    CU(launch_pairs_emit(st, r.o_sel, r.kl, r.keys, ids, r.o_a, r.o_b));
    return SVSB_OK;
}

static int top_pairs_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, int64_t n_pairs, float* out_scores,
                         int64_t* out_ids_a, int64_t* out_ids_b, int64_t* out_count) {
    if (!out_count) return fail(SVSB_E_INVALID, "svsb_top_pairs: out_count is NULL");
    *out_count = 0;
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident (call svsb_load_* first)");
    const int64_t N = g->n;
    if (n_pairs <= 0 || N < 2 || g->d == 0) return SVSB_OK;       // get_top_k: k <= 0 -> [] (util.py:200-201); no pairs
    if (!out_scores || !out_ids_a || !out_ids_b) return fail(SVSB_E_INVALID, "svsb_top_pairs: NULL buffer");
    if (g->has_tombstones()) return fail(SVSB_E_INVALID, "svsb_top_pairs: the resident generation has tombstoned rows (reload to compact it)");
    if (N > 0x7fffff00ll) return fail(SVSB_E_INVALID, "svsb_top_pairs: too many rows");
    const float R = 1.0f + g->max_dev;
    if (!(R <= 8.0f)) return fail(SVSB_E_INVALID, "svsb_top_pairs: rows are too far from unit norm for the fp16 coarse pass");
    const double total_pairs = 0.5 * (double)N * (double)(N - 1);
    const int64_t n = (double)n_pairs < total_pairs ? n_pairs : (int64_t)total_pairs;       // util.py:198-199
    if (n > (1ll << 22)) return fail(SVSB_E_INVALID, "svsb_top_pairs: at most 2^22 pairs per call");
    const float eps2 = pairs_eps2(g->d, R);
    if (e->multi) return multi_top_pairs(e, g, n, eps2, out_scores, out_ids_a, out_ids_b, out_count);

    std::lock_guard<std::mutex> lk(e->batch_mu);
    const PairRows rows = pair_rows_of({g.get()});
    PairsDev r;
    int rc;
    if ((rc = pairs_dev_prepare(e, g.get(), n, eps2, r)) != SVSB_OK) return rc;
    if ((rc = pairs_dev_coarse(r, 0, pairs_plan({N})[0], {PairShadow{g->M16, g->shards[0].dev}}, rows)) != SVSB_OK) return rc;
    if (r.C < n) return fail(SVSB_E_CUDA, "internal: pair list shorter than the requested count");
    if ((rc = pairs_dev_alloc(r)) != SVSB_OK) return rc;
    if ((rc = pairs_dev_finish(r, rows, g->shards[0].ids)) != SVSB_OK) return rc;
    CU(cudaMemcpyAsync(out_scores, r.o_scores, (size_t)n * 4, cudaMemcpyDeviceToHost, r.st));
    CU(cudaMemcpyAsync(out_ids_a, r.o_a, (size_t)n * 8, cudaMemcpyDeviceToHost, r.st));
    CU(cudaMemcpyAsync(out_ids_b, r.o_b, (size_t)n * 8, cudaMemcpyDeviceToHost, r.st));
    CU(cudaStreamSynchronize(r.st));
    *out_count = n;
    return SVSB_OK;
}

extern "C" int svsb_top_pairs(svsb_t* e, int64_t n_pairs, float* out_scores, int64_t* out_ids_a, int64_t* out_ids_b,
                              int64_t* out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    return top_pairs_gen(e, pin(e), n_pairs, out_scores, out_ids_a, out_ids_b, out_count);
}
extern "C" int svsb_snapshot_top_pairs(svsb_t* e, svsb_snap_t* s, int64_t n_pairs, float* out_scores, int64_t* out_ids_a,
                                       int64_t* out_ids_b, int64_t* out_count) {
    if (!e || !s) return fail(SVSB_E_INVALID, "svsb_snapshot_top_pairs: NULL argument");
    return top_pairs_gen(e, s->gen, n_pairs, out_scores, out_ids_a, out_ids_b, out_count);
}

// ---- peer memory of the one-process-per-GPU deployment: what a rank maps of its peers, and when it lets go -----------
// The query exchange (Xchg), the batch window (BXchg) and the pair search (PairsShard) read or write other ranks' device
// memory.  A connect that fails part-way closes what it opened; an unmap leaves the state create left.
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");

int PeerMaps::open(const void* handle, void** out, const char* who) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    const cudaError_t ce = cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess);
    (void)cudaGetLastError();
    if (ce != cudaSuccess) return fail(SVSB_E_CUDA, std::string(who) + ": cudaIpcOpenMemHandle: " + cudaGetErrorString(ce));
    opened.push_back(*out);
    return SVSB_OK;
}

int PeerMaps::reach(int self, int dev, const char* who) {
    if (dev == self) return SVSB_OK;
    int can = 0;
    CU(cudaDeviceCanAccessPeer(&can, self, dev));
    if (!can) return fail(SVSB_E_CUDA, std::string(who) + ": no peer access between the devices");
    const cudaError_t pe = cudaDeviceEnablePeerAccess(dev, 0);
    (void)cudaGetLastError();
    if (pe == cudaSuccess || pe == cudaErrorPeerAccessAlreadyEnabled) return SVSB_OK;    // another connect enabled it before
    return fail(SVSB_E_CUDA, std::string(who) + ": enabling peer access: " + cudaGetErrorString(pe));
}

void PeerMaps::close() {
    for (void* p : opened) cudaIpcCloseMemHandle(p);
    opened.clear();
}

int PeerWindow::publish(void* handle_out) {
    peer_block.assign(world, nullptr);
    peer_block[rank] = block;
    if (const char* v = getenv("SVSB_XCHG_TIMEOUT_MS")) { const long long ms = atoll(v); if (ms > 0) timeout_ns = (unsigned long long)ms * 1000000ull; }
    if (handle_out) {
        cudaIpcMemHandle_t h;
        CU(cudaIpcGetMemHandle(&h, block));
        memcpy(handle_out, &h, 64);
    }
    connected = world == 1;
    return SVSB_OK;
}

int PeerWindow::connect(const void* handles, const char* who) {
    for (int r = 0; r < world; ++r) {
        if (r == rank) continue;
        void* p = nullptr;
        const int rc = maps.open(static_cast<const unsigned char*>(handles) + (size_t)r * 64, &p, who);
        if (rc != SVSB_OK) { unmap(); return rc; }
        peer_block[r] = static_cast<unsigned char*>(p);
    }
    connected = true;
    return SVSB_OK;
}

int PeerWindow::connect_local(int dev, svsb_engine* const* engines, PeerWindow* (*window_of)(svsb_engine*, const PeerWindow*),
                              const char* who) {
    for (int r = 0; r < world; ++r) {
        if (r == rank) continue;
        svsb_engine* o = engines[r];
        const PeerWindow* w = o ? window_of(o, this) : nullptr;
        if (!w || w->world != world || w->rank != r) { unmap(); return fail(SVSB_E_INVALID, std::string(who) + ": peer engine has no matching window"); }
        const int rc = maps.reach(dev, o->devs[0], who);
        if (rc != SVSB_OK) { unmap(); return rc; }
        peer_block[r] = w->block;
    }
    connected = true;
    return SVSB_OK;
}

void PeerWindow::unmap() {
    maps.close();
    for (size_t r = 0; r < peer_block.size(); ++r) if ((int)r != rank) peer_block[r] = nullptr;
    connected = world == 1;
}

// world / rank of a protocol of the one-process-per-GPU deployment, on an engine of one device
static int check_world_rank(const svsb_engine* e, int32_t world, int32_t rank, const char* who) {
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, std::string(who) + ": a sharded engine owns exactly one device");
    if (world < 1 || world > XCHG_MAX_RANKS || rank < 0 || rank >= world)
        return fail(SVSB_E_INVALID, std::string(who) + ": bad world / rank (<= 16 ranks)");
    return SVSB_OK;
}

// ---- pairwise top pairs of the one-process-per-GPU deployment (include/svsb200.h svsb_pairs_*) ----------------------
// Rank r runs pairs_plan(shard rows)[r] -- the same per-device pass as multi_top_pairs -- against its peers' shards opened
// over CUDA IPC; the caller all-gathers the per-rank lists and every rank merges them.
constexpr uint32_t PAIRS_DESC_MAGIC = 0x53505231u;
struct PairsDesc {                                 // svsb_pairs_export's descriptor (SVSB_PAIRS_DESC_BYTES)
    uint32_t magic = 0; int32_t has_rows = 0;      // has_rows = 0: an empty shard, no handles
    int64_t n = 0, row0 = 0;
    uint64_t gen = 0;
    int32_t d = 0, ld = 0, ld16 = 0, pad = 0;
    cudaIpcMemHandle_t M, M16, ids;                // fp32 rows, fp16 shadow, embeddings.id
};
static_assert(sizeof(PairsDesc) <= SVSB_PAIRS_DESC_BYTES, "pair descriptor does not fit");

// one rank's shard as connect sees it
struct PairsPeer { int64_t n = 0, row0 = 0; int d = 0, ld = 0; const float* M = nullptr; const void* M16 = nullptr; const int64_t* ids = nullptr; };

static void pairs_unmap(PairsShard* p) {
    p->maps.close();
    p->connected = false;
}

static void pairs_release(svsb_engine* e) {
    PairsShard* p = e->pairs.get();
    if (!p) return;
    cudaSetDevice(e->devs[0]);
    pairs_unmap(p);
    if (p->ev) cudaEventDestroy(p->ev);
    e->pairs.reset();
}

static PairsPeer pairs_peer_of(const Generation* g) {
    const Shard& s = g->shards[0];
    PairsPeer q; q.n = s.n; q.row0 = s.row0; q.d = g->d; q.ld = g->ld; q.M = s.M; q.M16 = g->M16; q.ids = s.ids;
    return q;
}

extern "C" int svsb_pairs_export(svsb_t* e, float* max_dev_out, int64_t* rows_out, void* desc_out) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!desc_out) return fail(SVSB_E_INVALID, "svsb_pairs_export: NULL descriptor");
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, "svsb_pairs_export: a sharded engine owns exactly one device");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident (call svsb_load_* first)");
    if (g->has_tombstones()) return fail(SVSB_E_INVALID, "svsb_top_pairs: the resident generation has tombstoned rows (reload to compact it)");
    std::lock_guard<std::mutex> lk(e->batch_mu);
    if (e->pairs && e->pairs->connected) return fail(SVSB_E_STATE, "svsb_pairs_export: svsb_pairs_disconnect first");
    CU(cudaSetDevice(e->devs[0]));
    if (!e->pairs) {
        std::unique_ptr<PairsShard> p(new PairsShard());
        CU(cudaEventCreateWithFlags(&p->ev, cudaEventDisableTiming));
        e->pairs = std::move(p);
    }
    const Shard& s = g->shards[0];
    PairsDesc D;
    D.magic = PAIRS_DESC_MAGIC; D.n = s.n; D.row0 = s.row0; D.gen = g->id; D.d = g->d; D.ld = g->ld; D.ld16 = (g->d + 7) & ~7;
    memset(&D.M, 0, 64); memset(&D.M16, 0, 64); memset(&D.ids, 0, 64);
    if (s.n > 0 && s.M) {                          // the fp16 shadow the peers' rectangle tasks copy blocks of
        BatchWs* w = nullptr;
        int rc = batch_ws_get(e, w);
        if (rc != SVSB_OK) return rc;
        BatchPlan P; P.ld16 = D.ld16;
        if ((rc = ensure_m16(g.get(), P, w->st)) != SVSB_OK) return rc;
        CU(cudaIpcGetMemHandle(&D.M, s.M));
        CU(cudaIpcGetMemHandle(&D.M16, g->M16));
        CU(cudaIpcGetMemHandle(&D.ids, s.ids));
        D.has_rows = 1;
    }
    e->pairs->gen = g;                             // the previous export's generation is released here
    memset(desc_out, 0, SVSB_PAIRS_DESC_BYTES);
    memcpy(desc_out, &D, sizeof(D));
    if (max_dev_out) *max_dev_out = g->max_dev;
    if (rows_out) *rows_out = s.n;
    return SVSB_OK;
}

// Check the ranks' shards (peers[rank] is this rank's own) and build the tables of the pass and the merge.
static int pairs_finish_connect(PairsShard* p, int world, int rank, const std::vector<PairsPeer>& peers, const char* who) {
    int d = -1, ld = -1;
    for (int r = 0; r < world; ++r) {
        const PairsPeer& q = peers[(size_t)r];
        if (r + 1 < world && peers[(size_t)r + 1].row0 != q.row0 + q.n)
            return fail(SVSB_E_INVALID, std::string(who) + ": the ranks' row ranges are not contiguous in rank order");
        if (q.n == 0 || q.d == 0) continue;
        if (!q.M || !q.M16 || !q.ids) return fail(SVSB_E_INVALID, std::string(who) + ": a rank exported rows without buffers");
        if (d < 0) { d = q.d; ld = q.ld; }
        else if (q.d != d || q.ld != ld) return fail(SVSB_E_INVALID, std::string(who) + ": the ranks' row widths (d, ld) differ");
    }
    PairRows t;
    t.n = world;
    for (int r = 0; r < world; ++r) {
        t.row0[r] = peers[(size_t)r].row0 - peers[0].row0; t.M[r] = peers[(size_t)r].M; t.ids[r] = peers[(size_t)r].ids;
    }
    t.row0[world] = t.row0[world - 1] + peers[(size_t)world - 1].n;
    p->rows = t;
    p->world = world; p->rank = rank; p->d = d < 0 ? 0 : d;
    p->shard_rows.clear(); p->shadows.clear();
    for (const PairsPeer& q : peers) { p->shard_rows.push_back(q.n); p->shadows.push_back(PairShadow{q.M16, -1}); }
    p->connected = true;
    return SVSB_OK;
}

static int pairs_connect_check(svsb_engine* e, int32_t world, int32_t rank, const void* arg, const char* who) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!arg) return fail(SVSB_E_INVALID, std::string(who) + ": NULL argument");
    if (!e->pairs || !e->pairs->gen) return fail(SVSB_E_STATE, std::string(who) + ": svsb_pairs_export first");
    if (e->pairs->connected) return fail(SVSB_E_STATE, std::string(who) + ": already connected (svsb_pairs_disconnect first)");
    return check_world_rank(e, world, rank, who);
}

extern "C" int svsb_pairs_connect(svsb_t* e, int32_t world, int32_t rank, const void* descs) {
    int rc = pairs_connect_check(e, world, rank, descs, "svsb_pairs_connect");
    if (rc != SVSB_OK) return rc;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    PairsShard* p = e->pairs.get();
    CU(cudaSetDevice(e->devs[0]));
    std::vector<PairsPeer> peers((size_t)world);
    for (int r = 0; r < world; ++r) {
        if (r == rank) { peers[(size_t)r] = pairs_peer_of(p->gen.get()); continue; }
        PairsDesc D;
        memcpy(&D, static_cast<const unsigned char*>(descs) + (size_t)r * SVSB_PAIRS_DESC_BYTES, sizeof(D));
        if (D.magic != PAIRS_DESC_MAGIC) { pairs_unmap(p); return fail(SVSB_E_INVALID, "svsb_pairs_connect: not a svsb_pairs_export descriptor"); }
        PairsPeer& q = peers[(size_t)r];
        q.n = D.n; q.row0 = D.row0; q.d = D.d; q.ld = D.ld;
        if (!D.has_rows) continue;
        void* ptr[3] = {nullptr, nullptr, nullptr};
        const cudaIpcMemHandle_t* h[3] = {&D.M, &D.M16, &D.ids};
        for (int i = 0; i < 3; ++i)
            if ((rc = p->maps.open(h[i], &ptr[i], "svsb_pairs_connect")) != SVSB_OK) { pairs_unmap(p); return rc; }
        q.M = static_cast<const float*>(ptr[0]); q.M16 = ptr[1]; q.ids = static_cast<const int64_t*>(ptr[2]);
    }
    if ((rc = pairs_finish_connect(p, world, rank, peers, "svsb_pairs_connect")) != SVSB_OK) pairs_unmap(p);
    return rc;
}

extern "C" int svsb_pairs_connect_local(svsb_t* e, int32_t world, int32_t rank, svsb_t* const* engines) {
    int rc = pairs_connect_check(e, world, rank, engines, "svsb_pairs_connect_local");
    if (rc != SVSB_OK) return rc;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    PairsShard* p = e->pairs.get();
    CU(cudaSetDevice(e->devs[0]));
    std::vector<PairsPeer> peers((size_t)world);
    for (int r = 0; r < world; ++r) {
        svsb_engine* o = r == rank ? e : engines[r];
        if (!o || !o->pairs || !o->pairs->gen)
            return fail(SVSB_E_INVALID, "svsb_pairs_connect_local: a peer engine has not exported (svsb_pairs_export)");
        // the re-score and the merge read the peer's rows and ids directly
        if ((rc = p->maps.reach(e->devs[0], o->devs[0], "svsb_pairs_connect_local")) != SVSB_OK) return rc;
        peers[(size_t)r] = pairs_peer_of(o->pairs->gen.get());
    }
    return pairs_finish_connect(p, world, rank, peers, "svsb_pairs_connect_local");
}

extern "C" int svsb_pairs_local(svsb_t* e, void* stream, int64_t n_pairs, float max_row_norm, float* d_scores, int64_t* d_rows_a,
                                int64_t* d_rows_b, int64_t* out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!out_count) return fail(SVSB_E_INVALID, "svsb_pairs_local: out_count is NULL");
    *out_count = 0;
    PairsShard* p = e->pairs.get();
    if (!p || !p->connected) return fail(SVSB_E_STATE, "svsb_pairs_local: svsb_pairs_connect first");
    const int64_t N = p->rows.row0[p->world];
    if (n_pairs <= 0 || N < 2 || p->d == 0) return SVSB_OK;
    if (!d_scores || !d_rows_a || !d_rows_b) return fail(SVSB_E_INVALID, "svsb_pairs_local: NULL buffer");
    if (N > 0x7fffff00ll) return fail(SVSB_E_INVALID, "svsb_top_pairs: too many rows");
    const float R = max_row_norm;
    if (!(R <= 8.0f)) return fail(SVSB_E_INVALID, "svsb_top_pairs: rows are too far from unit norm for the fp16 coarse pass");
    const double total_pairs = 0.5 * (double)N * (double)(N - 1);
    const int64_t n = (double)n_pairs < total_pairs ? n_pairs : (int64_t)total_pairs;
    if (n > (1ll << 22)) return fail(SVSB_E_INVALID, "svsb_top_pairs: at most 2^22 pairs per call");
    const float eps2 = pairs_eps2(p->d, R);

    std::lock_guard<std::mutex> lk(e->batch_mu);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    PairsDev r;
    int rc;
    if ((rc = pairs_dev_prepare(e, p->gen.get(), n, eps2, r)) != SVSB_OK) return rc;
    if (!r.w) return SVSB_OK;                      // no rows on this rank: its share of the plan is empty
    CU(cudaEventRecord(p->ev, st));                // the caller's outputs are written behind what its stream already holds
    CU(cudaStreamWaitEvent(r.st, p->ev, 0));
    if ((rc = pairs_dev_coarse(r, p->rank, pairs_plan(p->shard_rows)[(size_t)p->rank], p->shadows, p->rows)) != SVSB_OK) return rc;
    if ((rc = pairs_dev_alloc(r)) != SVSB_OK) return rc;
    if (r.kl == 0) return SVSB_OK;
    if ((rc = pairs_dev_finish(r, p->rows, nullptr)) != SVSB_OK) return rc;          // global rows: the merge maps them to ids
    CU(cudaMemcpyAsync(d_scores, r.o_scores, (size_t)r.kl * 4, cudaMemcpyDeviceToDevice, r.st));
    CU(cudaMemcpyAsync(d_rows_a, r.o_a, (size_t)r.kl * 8, cudaMemcpyDeviceToDevice, r.st));
    CU(cudaMemcpyAsync(d_rows_b, r.o_b, (size_t)r.kl * 8, cudaMemcpyDeviceToDevice, r.st));
    CU(cudaStreamSynchronize(r.st));
    *out_count = r.kl;
    return SVSB_OK;
}

extern "C" int svsb_pairs_merge(svsb_t* e, void* stream, const float* d_scores, const int64_t* d_rows_a, const int64_t* d_rows_b,
                                const int32_t* d_counts, int32_t world, int64_t stride, int64_t n, float* d_out_scores,
                                int64_t* d_out_ids_a, int64_t* d_out_ids_b, int32_t* d_out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    PairsShard* p = e->pairs.get();
    if (!p || !p->connected) return fail(SVSB_E_STATE, "svsb_pairs_merge: svsb_pairs_connect first");
    if (world != p->world) return fail(SVSB_E_INVALID, "svsb_pairs_merge: world differs from the connected one");
    if (stride < 1 || n < 1 || n > (1ll << 22)) return fail(SVSB_E_INVALID, "svsb_pairs_merge: stride >= 1, 1 <= n <= 2^22");
    if (!d_scores || !d_rows_a || !d_rows_b || !d_counts || !d_out_scores || !d_out_ids_a || !d_out_ids_b || !d_out_count)
        return fail(SVSB_E_INVALID, "svsb_pairs_merge: NULL buffer");
    CU(cudaSetDevice(e->devs[0]));
    CU(launch_merge_sorted_pairs(static_cast<cudaStream_t>(stream), d_scores, d_rows_a, d_rows_b, d_counts, world, stride, n, p->rows,
                                 d_out_scores, d_out_ids_a, d_out_ids_b, d_out_count));
    return SVSB_OK;
}

extern "C" int svsb_pairs_disconnect(svsb_t* e) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    PairsShard* p = e->pairs.get();
    if (!p) return SVSB_OK;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    CU(cudaSetDevice(e->devs[0]));
    pairs_unmap(p);
    p->gen.reset();
    return SVSB_OK;
}

// Diagnostics of the last svsb_query_batch / svsb_bench_run_batch chunk: per query the number of coarse candidates,
// the number of rows re-scored exactly, and the flag word (0 = answered by the coarse path).
extern "C" int svsb_batch_stats(svsb_t* e, int32_t b, int32_t* candidates, int32_t* rescored, int32_t* flags) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = e->batch_ws.get();
    if (!w || b < 0 || b > w->cap_b) return fail(SVSB_E_STATE, "svsb_batch_stats: no batch of that size has run");
    CU(cudaSetDevice(w->dev));
    CU(cudaStreamSynchronize(w->st));
    if (candidates) CU(cudaMemcpy(candidates, w->cand_cnt, (size_t)b * 4, cudaMemcpyDeviceToHost));
    if (rescored) CU(cudaMemcpy(rescored, w->stats, (size_t)b * 4, cudaMemcpyDeviceToHost));
    if (flags) CU(cudaMemcpy(flags, w->flags, (size_t)b * 4, cudaMemcpyDeviceToHost));
    return SVSB_OK;
}

// Diagnostics: query q's coarse candidate list of the last chunk (keys make_key(coarse score, row), in the order the
// coarse pass appended them), its full count (above the list's capacity when the list overflowed) and its eps.  The
// refine kernels only read the lists, so they are intact after the batch has been answered.
extern "C" int svsb_batch_candidates(svsb_t* e, int32_t q, int64_t cap, uint64_t* keys, int32_t* count, float* eps) {
    if (!e || !count) return fail(SVSB_E_INVALID, "svsb_batch_candidates: NULL argument");
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = e->batch_ws.get();
    if (!w || q < 0 || q >= w->cap_b || !w->cand) return fail(SVSB_E_STATE, "svsb_batch_candidates: no batch has run with that query");
    CU(cudaSetDevice(w->dev));
    CU(cudaStreamSynchronize(w->st));
    int32_t cnt = 0;
    CU(cudaMemcpy(&cnt, w->cand_cnt + q, 4, cudaMemcpyDeviceToHost));
    *count = cnt;
    const int64_t m = std::min<int64_t>(std::min<int64_t>(cnt, w->cand_cap), std::max<int64_t>(cap, 0));
    if (keys && m > 0) CU(cudaMemcpy(keys, w->cand + (size_t)q * w->cand_cap, (size_t)m * 8, cudaMemcpyDeviceToHost));
    if (eps) CU(cudaMemcpy(eps, w->eps + q, 4, cudaMemcpyDeviceToHost));
    return SVSB_OK;
}

extern "C" int svsb_batch_threshold_mode(svsb_t* e) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    return (g->batch_guaranteed.load(std::memory_order_relaxed) || env_int("SVSB_BATCH_GUARANTEED", 0) != 0) ? 1 : 0;
}

extern "C" int svsb_topk_scores(svsb_t* e, const float* scores, int64_t n, int32_t k,
                                float* out_scores, int64_t* out_index, int32_t* out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!out_count) return fail(SVSB_E_INVALID, "svsb_topk_scores: out_count is NULL");
    *out_count = 0;
    if (n < 0) return fail(SVSB_E_INVALID, "svsb_topk_scores: negative n");
    if (n > 0xfffffff0ll) return fail(SVSB_E_INVALID, "svsb_topk_scores: more than 2^32 scores");
    const int64_t kk = std::min<int64_t>(k, n);
    if (kk <= 0) return SVSB_OK;
    if (!scores || !out_scores || !out_index) return fail(SVSB_E_INVALID, "svsb_topk_scores: NULL buffer");
    CtxLease lease(e);
    int rc = ctx_acquire(e, lease.c);
    if (rc != SVSB_OK) return rc;
    QueryCtx* c = lease.c.get();
    DevWs& w = c->ws[0];
    if ((rc = ctx_ensure_host(c, 4, kk)) != SVSB_OK) return rc;
    if ((rc = w.ensure_query(n, std::max<int64_t>(kk, 128), kk)) != SVSB_OK) return rc;
    CU(cudaSetDevice(w.dev));
    Shard rows; rows.n = rows.n_live = n;                         // no ids: the selection returns rows
    CU(cudaMemcpyAsync(w.scores, scores, (size_t)n * 4, cudaMemcpyHostToDevice, w.st));
    if (kk <= K_FAST_MAX) CU(launch_groupmax(w.st, w.dev, w.scores, n, w.gmax, group_shift_for(n)));
    if ((rc = select_phase(w.st, w, nullptr, rows, nullptr, 0, kk, w.out())) != SVSB_OK) return rc;
    CU(cudaMemcpyAsync(c->h_scores, w.out_scores, (size_t)kk * 4, cudaMemcpyDeviceToHost, w.st));
    CU(cudaMemcpyAsync(c->h_ids, w.out_ids, (size_t)kk * 8, cudaMemcpyDeviceToHost, w.st));
    CU(cudaMemcpyAsync(c->h_count, w.out_count, 4, cudaMemcpyDeviceToHost, w.st));
    CU(cudaStreamSynchronize(w.st));
    memcpy(out_scores, c->h_scores, (size_t)kk * 4);
    memcpy(out_index, c->h_ids, (size_t)kk * 8);
    *out_count = *c->h_count;
    return SVSB_OK;
}

// ------------------------------------------------------------------------------------------------
// measurement support
// ------------------------------------------------------------------------------------------------
extern "C" int svsb_bench_set_queries(svsb_t* e, const float* Q, int32_t nq, int32_t d) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!Q || nq <= 0 || d <= 0) return fail(SVSB_E_INVALID, "svsb_bench_set_queries: bad arguments");
    const int ld = round_up4(d);
    std::vector<float> padded((size_t)nq * ld, 0.f);
    stage_queries(padded.data(), Q, nq, d, ld);
    if (e->bench_q.size() != e->devs.size()) e->bench_q.assign(e->devs.size(), nullptr);
    for (size_t i = 0; i < e->devs.size(); ++i) {
        CU(cudaSetDevice(e->devs[i]));
        if (e->bench_q[i]) { cudaFree(e->bench_q[i]); e->bench_q[i] = nullptr; }
        CU(cudaMalloc(&e->bench_q[i], padded.size() * 4));
        CU(cudaMemcpy(e->bench_q[i], padded.data(), padded.size() * 4, cudaMemcpyHostToDevice));
    }
    e->bench_nq = nq; e->bench_d = d; e->bench_ld = ld;
    return SVSB_OK;
}

// Timing events for the similarity kernel inside the timed loop: owned by the engine, created on ITS device 0.
static int ensure_kernel_events(svsb_engine* e, int dev, size_t n) {
    CU(cudaSetDevice(dev));
    while (e->bench_kev.size() < n) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); e->bench_kev.push_back(ev); }
    return SVSB_OK;
}

extern "C" int svsb_bench_run(svsb_t* e, int32_t k, int32_t iters, float* total_ms, float* gemv_ms, int64_t* launches) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (e->bench_nq == 0 || e->bench_d != g->d) return fail(SVSB_E_SHAPE, "svsb_bench_run: upload queries of the matrix's d first");
    if (k <= 0 || iters <= 0 || g->n_live == 0) return fail(SVSB_E_INVALID, "svsb_bench_run: bad arguments");
    const int64_t kk = std::min<int64_t>(k, g->n_live);
    const int64_t l0 = g_launches.load();
    int rc;
    if (e->multi) {                                     // several devices: the fused path with its tickets in flight (multi.cu)
        rc = multi_bench_run(e, g, k, iters, total_ms, gemv_ms);
        if (launches) *launches = g_launches.load() - l0;
        return rc;
    }
    if (!e->bench_ctx) { if ((rc = ctx_create(e, e->bench_ctx)) != SVSB_OK) return rc; }
    QueryCtx* c = e->bench_ctx.get();
    DevWs& w0 = c->ws[0];
    const Shard& s = g->shards[0];
    if ((rc = prepare_ws(w0, g.get(), s, kk)) != SVSB_OK) return rc;
    // gemv_ms requested: bracket similarity-kernel launches with events INSIDE the timed loop (one launch in
    // KTIME_EVERY: the two event records cost ~5 us of stream time per bracketed launch, 4 % of a 125 k-row shard's
    // query -- profiles/r01_shard_probe.txt -- and the loop being timed should be the product's)
    const bool ktime = gemv_ms != nullptr;
    constexpr int KTIME_EVERY = 8;
    auto timed_it = [&](int it) { return ktime && it % KTIME_EVERY == 0; };
    if (ktime && (rc = ensure_kernel_events(e, w0.dev, (size_t)iters * 2)) != SVSB_OK) return rc;
    // k <= 2048: software pipeline.  The similarity kernel of query i+1 (stream A, all SMs but one) runs while the
    // one-CTA selection kernel of query i (stream B) finishes on the SM left free; two buffer sets.
    const bool pipelined = kk <= K_FAST_MAX && env_int("SVSB_PIPELINE", 1) != 0 && sm_count(w0.dev) > 8;
    const int route = filter_route(s, kk);
    e->bench_route = route;
    if (pipelined) {
        if (!c->alt) {
            c->alt.reset(new DevWs());
            DevWs& a = *c->alt;
            a.dev = w0.dev;
            CU(cudaSetDevice(a.dev));
            CU(cudaStreamCreateWithFlags(&a.st, cudaStreamNonBlocking));
            a.own_stream = true;
            CU(cudaEventCreateWithFlags(&a.ev, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&a.ev_sel, cudaEventDisableTiming));
        }
        if ((rc = prepare_ws(*c->alt, g.get(), s, kk)) != SVSB_OK) return rc;
    }
    std::vector<cudaEvent_t>& kev = e->bench_kev;
    CU(cudaSetDevice(w0.dev));
    CU(cudaStreamSynchronize(w0.st));
    if (pipelined) CU(cudaStreamSynchronize(c->alt->st));
    CU(cudaEventRecord(w0.ev0, w0.st));
    for (int it = 0; it < iters; ++it) {
        DevWs& W = (pipelined && (it & 1)) ? *c->alt : w0;
        cudaStream_t sb = pipelined ? c->alt->st : w0.st;           // the selections' stream
        const float* q = e->bench_q[0] + (int64_t)(it % e->bench_nq) * e->bench_ld;
        if (pipelined && it >= 2) CU(cudaStreamWaitEvent(w0.st, W.ev_sel, 0));   // selection of query it-2 is done with W
        cudaEvent_t* t = timed_it(it) ? &kev[2 * it] : nullptr;
        if ((rc = similarity_phase(w0.st, W, g.get(), s, q, route, pipelined ? 1 : 0, false, t)) != SVSB_OK) return rc;
        if (pipelined && (rc = W.hand_off(w0.st, sb)) != SVSB_OK) return rc;
        if ((rc = select_phase(sb, W, g.get(), s, q, route, kk, W.out())) != SVSB_OK) return rc;
        if (pipelined) CU(cudaEventRecord(W.ev_sel, sb));
        c->last = &W;
    }
    if (pipelined) {
        CU(cudaStreamWaitEvent(w0.st, w0.ev_sel, 0));
        if (iters > 1) CU(cudaStreamWaitEvent(w0.st, c->alt->ev_sel, 0));
    }
    CU(cudaEventRecord(w0.ev1, w0.st));
    CU(cudaEventSynchronize(w0.ev1));
    float ms = 0.f; CU(cudaEventElapsedTime(&ms, w0.ev0, w0.ev1));
    if (total_ms) *total_ms = ms;
    if (launches) *launches = g_launches.load() - l0;
    if (ktime) {
        float sum = 0.f; int cnt = 0;
        for (int it = 0; it < iters; ++it)
            if (timed_it(it)) { float t = 0.f; CU(cudaEventElapsedTime(&t, kev[2 * it], kev[2 * it + 1])); sum += t; ++cnt; }
        *gemv_ms = sum * (float)iters / (float)cnt;            // mean bracketed launch x launches
    } else if (gemv_ms) *gemv_ms = 0.f;
    return SVSB_OK;
}

extern "C" int svsb_bench_filter_stats(svsb_t* e, int32_t* filter, int64_t* rescored) {
    if (!e || !filter || !rescored) return fail(SVSB_E_INVALID, "svsb_bench_filter_stats: NULL argument");
    *filter = 0; *rescored = 0;
    if (e->multi || !e->bench_ctx || !e->bench_ctx->last) return SVSB_OK;
    if (!e->bench_route) return SVSB_OK;
    const DevWs& w = *e->bench_ctx->last;
    uint32_t st[2] = {0, 0};
    CU(cudaSetDevice(w.dev));
    CU(cudaStreamSynchronize(w.st));
    CU(cudaMemcpy(st, w.fstate, 8, cudaMemcpyDeviceToHost));
    *filter = 1; *rescored = st[1];
    return SVSB_OK;
}

extern "C" int svsb_bench_filter_route(svsb_t* e, int32_t* route) {
    if (!e || !route) return fail(SVSB_E_INVALID, "svsb_bench_filter_route: NULL argument");
    *route = e->multi || !e->bench_ctx || !e->bench_ctx->last ? 0 : e->bench_route;
    return SVSB_OK;
}

// Phase timestamps (ns, %globaltimer) of one selection-kernel run on the resident matrix with uploaded
// query `qi`: stamps[0..6] = entry, keys staged, threshold found, hit list, candidates, sorted, done;
// stamps[8] = candidate count, stamps[9] = groups rescanned.  Development aid for profiles/.
extern "C" int svsb_debug_select_phases(svsb_t* e, int32_t qi, int32_t k, uint64_t* stamps16) {
    if (!e || !stamps16) return fail(SVSB_E_INVALID, "svsb_debug_select_phases: NULL argument");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (e->bench_nq == 0 || qi < 0 || qi >= e->bench_nq || k < 1 || k > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_debug_select_phases: bad arguments");
    int rc;
    if (!e->bench_ctx) { if ((rc = ctx_create(e, e->bench_ctx)) != SVSB_OK) return rc; }
    DevWs& w = e->bench_ctx->ws[0];
    const Shard& s = g->shards[0];
    const int64_t kk = std::min<int64_t>(k, s.n_live);
    if (kk < 1) return fail(SVSB_E_INVALID, "svsb_debug_select_phases: no live rows");
    if ((rc = prepare_ws(w, g.get(), s, kk)) != SVSB_OK) return rc;
    CU(cudaSetDevice(w.dev));
    u64* dbg = nullptr;
    CU(cudaMalloc(&dbg, 16 * 8));
    CU(cudaMemsetAsync(dbg, 0, 16 * 8, w.st));
    const float* q = e->bench_q[0] + (int64_t)qi * e->bench_ld;
    if ((rc = similarity_phase(w.st, w, g.get(), s, q, 0)) != SVSB_OK) return rc;
    if ((rc = select_phase(w.st, w, g.get(), s, q, 0, kk, w.out(), dbg)) != SVSB_OK) return rc;
    CU(cudaMemcpyAsync(stamps16, dbg, 16 * 8, cudaMemcpyDeviceToHost, w.st));
    CU(cudaStreamSynchronize(w.st));
    CU(cudaFree(dbg));
    return SVSB_OK;
}

extern "C" int svsb_bench_run_batch(svsb_t* e, int32_t k, int32_t iters, float* total_ms, float* coarse_ms, int64_t* launches) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (e->bench_nq == 0 || e->bench_d != g->d) return fail(SVSB_E_SHAPE, "svsb_bench_run_batch: upload queries of the matrix's d first");
    if (k <= 0 || iters <= 0 || g->n_live == 0) return fail(SVSB_E_INVALID, "svsb_bench_run_batch: bad arguments");
    if (e->bench_nq > COARSE_MAX_BATCH) return fail(SVSB_E_INVALID, "svsb_bench_run_batch: at most 2048 uploaded queries");
    BatchPlan P;
    if (!batch_plan(e, g.get(), k, P)) return fail(SVSB_E_INVALID, "svsb_bench_run_batch: this matrix / k does not take the coarse path");
    const int b = e->bench_nq;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = nullptr;
    int rc = batch_acquire(e, g.get(), P, b, nullptr, w);
    if (rc != SVSB_OK) return rc;
    CU(cudaSetDevice(w->dev));
    const int64_t l0 = g_launches.load();
    CU(cudaStreamSynchronize(w->st));
    float csum = 0.f;
    CU(cudaEventRecord(w->ev[0], w->st));
    for (int it = 0; it < iters; ++it) {
        if ((rc = batch_enqueue(w, g.get(), P, e->bench_q[0], b, coarse_ms != nullptr, w->st)) != SVSB_OK) return rc;
        if (coarse_ms) {                                 // events are reused: collect before the next iteration records them
            CU(cudaEventSynchronize(w->ev[3]));
            float ms = 0.f; CU(cudaEventElapsedTime(&ms, w->ev[2], w->ev[3])); csum += ms;
        }
    }
    CU(cudaEventRecord(w->ev[1], w->st));
    CU(cudaEventSynchronize(w->ev[1]));
    float ms = 0.f; CU(cudaEventElapsedTime(&ms, w->ev[0], w->ev[1]));
    if (total_ms) *total_ms = ms;
    if (coarse_ms) *coarse_ms = csum;
    if (launches) *launches = g_launches.load() - l0;
    return SVSB_OK;
}

// Result of query qi of the last batch run (device-resident pipeline), for checking the timed path.
extern "C" int svsb_bench_batch_result(svsb_t* e, int32_t qi, int32_t k, float* out_scores, int64_t* out_emb_ids, int32_t* out_count,
                                       int32_t* out_flag) {
    if (!e || !out_scores || !out_emb_ids || !out_count) return fail(SVSB_E_INVALID, "svsb_bench_batch_result: NULL argument");
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = e->batch_ws.get();
    if (!w || qi < 0 || qi >= w->cap_b || k > w->cap_k) return fail(SVSB_E_STATE, "svsb_bench_batch_result: no such result");
    CU(cudaSetDevice(w->dev));
    CU(cudaStreamSynchronize(w->st));
    int32_t cnt = 0, flag = 0;
    CU(cudaMemcpy(&cnt, w->o_counts + qi, 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&flag, w->flags + qi, 4, cudaMemcpyDeviceToHost));
    if (cnt < 0 || cnt > k) return fail(SVSB_E_INVALID, "svsb_bench_batch_result: k does not match the run");
    CU(cudaMemcpy(out_scores, w->o_scores + (size_t)qi * k, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_emb_ids, w->o_ids + (size_t)qi * k, (size_t)cnt * 8, cudaMemcpyDeviceToHost));
    *out_count = cnt;
    if (out_flag) *out_flag = flag;
    return SVSB_OK;
}

extern "C" int svsb_bench_last_result(svsb_t* e, int32_t k, float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!out_scores || !out_emb_ids || !out_count) return fail(SVSB_E_INVALID, "svsb_bench_last_result: NULL buffer");
    if (e->multi) return multi_bench_last_result(e, k, out_scores, out_emb_ids, out_count);
    if (!e->bench_ctx || !e->bench_ctx->last) return fail(SVSB_E_STATE, "svsb_bench_last_result: no bench run yet");
    QueryCtx* c = e->bench_ctx.get();
    DevWs& w0 = *c->last;
    CU(cudaSetDevice(w0.dev));
    CU(cudaStreamSynchronize(c->ws[0].st));
    if (c->alt) CU(cudaStreamSynchronize(c->alt->st));
    int32_t cnt = 0;
    CU(cudaMemcpy(&cnt, w0.out_count, 4, cudaMemcpyDeviceToHost));
    if (cnt < 0 || cnt > k) return fail(SVSB_E_INVALID, "svsb_bench_last_result: k smaller than the result");
    CU(cudaMemcpy(out_scores, w0.out_scores, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_emb_ids, w0.out_ids, (size_t)cnt * 8, cudaMemcpyDeviceToHost));
    *out_count = cnt;
    return SVSB_OK;
}

// ------------------------------------------------------------------------------------------------
// sharded deployment: one process per GPU, the caller (torch.distributed) owns streams and the exchange
// ------------------------------------------------------------------------------------------------
extern "C" int svsb_set_shard(svsb_t* e, int64_t global_row0) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (global_row0 < 0) return fail(SVSB_E_INVALID, "svsb_set_shard: negative row offset");
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, "svsb_set_shard: a sharded engine owns exactly one device");
    e->shard_row0 = global_row0;
    return SVSB_OK;
}

// merge_records with the engine's merge scratch (slot 0's workspace holds it; only n_lists * cap > K_FAST_MAX needs it)
static int engine_merge_records(svsb_engine* e, cudaStream_t st, const RecordView& recs, int n_lists, int64_t list_words, int batch,
                                int k, float* out_scores, int64_t* out_ids, int32_t* out_counts, int verify_k, const int* status = nullptr) {
    u64* sk = nullptr; int64_t* sp = nullptr;
    if ((int64_t)n_lists * recs.cap > K_FAST_MAX) {
        DevWs& w = shard_slot(e, 0);
        int rc = w.ensure_merge_scratch((int64_t)batch * n_lists * recs.cap);
        if (rc != SVSB_OK) return rc;
        sk = w.mscr_keys; sp = w.mscr_ids;
    }
    return merge_records(st, recs, n_lists, list_words, batch, k, sk, sp, out_scores, out_ids, out_counts, verify_k, status);
}

static int enqueue_local_topk_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, void* stream, int32_t slot, const float* d_query,
                                  int32_t k, int64_t* d_record, int32_t flags);
extern "C" int svsb_enqueue_local_topk(svsb_t* e, void* stream, int32_t slot, const float* d_query, int32_t k,
                                       int64_t* d_record, int32_t flags) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    return enqueue_local_topk_gen(e, pin(e), stream, slot, d_query, k, d_record, flags);
}

// The next timing bracket of e->kev (svsb_kernel_time_collect), its two events created on first use.  The caller
// advances e->kev_used once the bracketed pass is enqueued.
static int kev_next(svsb_engine* e, cudaEvent_t*& t) {
    while (e->kev.size() < e->kev_used + 2) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); e->kev.push_back(ev); }
    t = &e->kev[e->kev_used];
    return SVSB_OK;
}

static int enqueue_local_topk_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, void* stream, int32_t slot, const float* d_query,
                                  int32_t k, int64_t* d_record, int32_t flags) {
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, "svsb_enqueue_local_topk: single-device engines only");
    if (slot < 0 || slot >= 8) return fail(SVSB_E_INVALID, "svsb_enqueue_local_topk: slot out of range (0..7)");
    if (k < 1) return fail(SVSB_E_INVALID, "svsb_enqueue_local_topk: k must be positive");
    if (!d_query || !d_record) return fail(SVSB_E_INVALID, "svsb_enqueue_local_topk: NULL pointer");
    const bool big = k > K_FAST_MAX;                        // full sort of the shard's keys, unpipelined (bit 1 ignored)
    const bool time_kernel = (flags & 1) != 0, pipelined = (flags & 2) != 0 && !big;
    const Shard& s = g->shards[0];
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaSetDevice(s.dev));
    const RecordView r{d_record, k};
    if (s.n_live == 0) { CU(cudaMemsetAsync(r.count(0), 0, 8, st)); return SVSB_OK; }
    DevWs& w = shard_slot(e, slot);
    int rc;
    if ((rc = w.ensure_query(s.n, std::max<int64_t>(std::min<int64_t>(k, s.n_live), K_FAST_MAX), k)) != SVSB_OK) return rc;
    if (pipelined) {
        if (!e->side_st) CU(cudaStreamCreateWithFlags(&e->side_st, cudaStreamNonBlocking));
        if (!w.ev) CU(cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming));
        if (!w.ev_sel) CU(cudaEventCreateWithFlags(&w.ev_sel, cudaEventDisableTiming));
    }
    // the slot's previous selection must have finished reading scores / group maxima before they are overwritten
    // (a plain call after a pipelined one on this slot, too)
    if ((rc = w.sel_wait(st)) != SVSB_OK) return rc;
    if (!pipelined) w.sel_pending = false;
    cudaEvent_t* t = nullptr;
    if (time_kernel && (rc = kev_next(e, t)) != SVSB_OK) return rc;
    // route 0 on purpose: filter_attach gives a one-process-per-GPU rank with enough rows the filter's shadows as well,
    // but only the single-device query paths take the filter (filter_route); the sharded and peer paths run K1
    if ((rc = similarity_phase(st, w, g.get(), s, d_query, 0, pipelined ? 1 : 0, false, t)) != SVSB_OK) return rc;
    if (t) e->kev_used += 2;
    if (pipelined && (rc = w.hand_off(st, e->side_st)) != SVSB_OK) return rc;
    if ((rc = select_phase(pipelined ? e->side_st : st, w, g.get(), s, d_query, 0, k, {r.keys(0), w.out_scores, r.ids(0), r.count(0)})) != SVSB_OK)
        return rc;
    if (pipelined) { CU(cudaEventRecord(w.ev_sel, e->side_st)); w.sel_pending = true; }
    return SVSB_OK;
}

// Batched form of svsb_enqueue_local_topk: local top-k records of b device-resident queries dQ[b][ld] (zero padded
// to the matrix's leading dimension) on the caller's stream, through the tensor-core coarse pass + exact refine where
// the shard / k allow it, else (and for queries the coarse pass flags) through the single-query kernels.  Synchronises
// `stream` once per <= 2048 queries to read the flag words.
extern "C" int svsb_batch_local_records(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, int64_t* d_records,
                                        int32_t* n_fallback) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    return batch_local_records_gen(e, pin(e), (cudaStream_t)stream, d_Q, b, k, d_records, n_fallback);
}

int batch_local_records_gen(svsb_engine* e, const std::shared_ptr<Generation>& g, cudaStream_t stream, const float* d_Q, int32_t b,
                            int32_t k, int64_t* d_records, int32_t* n_fallback) {
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, "svsb_batch_local_records: single-device engines only");
    if (b < 0 || k < 1 || k > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_batch_local_records: bad arguments (1 <= k <= 2048)");
    if (b == 0) return SVSB_OK;
    if (!d_Q || !d_records) return fail(SVSB_E_INVALID, "svsb_batch_local_records: NULL pointer");
    cudaStream_t st = stream;
    const RecordView recs{d_records, k};
    int fallbacks = 0;
    BatchPlan P;
    bool coarse = g->n_live > 0 && b >= env_int("SVSB_BATCH_MIN", 4) && batch_plan(e, g.get(), k, P);
    MqPlan MP;
    if (b >= 2 && mq_plan(g.get(), std::min<int64_t>(k, g->n_live), MP) && (b <= MP.max_b || !coarse)) {
        // small batch (or no tensor-core path for this shard): multi-query passes straight into the records
        std::lock_guard<std::mutex> lk(e->batch_mu);
        auto stage = [&](MqWs*, int c0, int, const float*& dQ) -> int { dQ = d_Q + (int64_t)c0 * g->ld; return SVSB_OK; };
        auto drain = [&](MqWs*, int c0, int) -> int {
            if (c0 + MP.chunk < b) CU(cudaStreamSynchronize(st));   // the next chunk reuses the score vectors
            return SVSB_OK;
        };
        int rc = mq_run(e, g.get(), MP, b, k, st, recs, stage, drain);
        if (rc != SVSB_OK) return rc;
        if (n_fallback) *n_fallback = 0;
        return SVSB_OK;
    }
    std::vector<char> todo((size_t)b, coarse ? 0 : 1);
    if (coarse) {
        std::lock_guard<std::mutex> lk(e->batch_mu);
        BatchWs* w = nullptr;
        int rc = batch_acquire(e, g.get(), P, std::min<int32_t>(b, COARSE_MAX_BATCH), st, w);
        if (rc == SVSB_E_NOMEM) std::fill(todo.begin(), todo.end(), 1);    // no room for the fp16 shadow (+50 % of the shard)
        else if (rc != SVSB_OK) return rc;                                 // or the workspace: the exact kernels answer, as in svsb_query_batch
        for (int32_t c0 = 0; rc == SVSB_OK && c0 < b; c0 += COARSE_MAX_BATCH) {
            const int bc = std::min<int32_t>(COARSE_MAX_BATCH, b - c0);
            const RefineOut o = recs.from(c0).refine_out();
            rc = batch_run_chunk(e, g.get(), P, w, st, d_Q + (int64_t)c0 * P.ld, bc, &o, [] { return SVSB_OK; });
            if (rc != SVSB_OK) return rc;
            for (int i = 0; i < bc; ++i) if (w->h_flags[i] != 0) todo[c0 + i] = 1;
        }
    }
    for (int32_t i = 0; i < b; ++i) {
        if (!todo[i]) continue;
        ++fallbacks;
        int rc = enqueue_local_topk_gen(e, g, stream, 0, d_Q + (int64_t)i * g->ld, k, recs.rec(i), 0);
        if (rc != SVSB_OK) return rc;
    }
    if (n_fallback) *n_fallback = fallbacks;
    return SVSB_OK;
}

// ---- sharded batches with a GLOBAL filter threshold (DESIGN.md section 6c) --------------------------------------------
// With local thresholds every rank finds ITS OWN top kk: it samples, filters and re-scores for a cut at local rank kk,
// although the shard holds only ~kk / world of the global top kk -- the fixed per-batch costs do not shrink with the
// shard (round 1: 31 % scaling efficiency at 8 GPUs).  Here the ranks agree on ONE threshold per query: each extracts the
// SAMPLE_TOPX largest coarse scores of its own sample (svsb_batch_sample_tops), the caller all-gathers those b x 32
// floats, and every rank takes the sample_rank-th largest of the UNION (svsb_batch_global_records) -- an order
// statistic of a sample of ALL rows, so the filter keeps ~(global rank sample_rank / f) / world rows per rank.  Every
// candidate is re-scored exactly; the record carries ver = #{coarse >= thr + 2 eps}; the merge adds ver over the ranks
// and accepts the query only if the sum reaches kk (then thr <= tau~_global - 2 eps: no rank's list misses a row of
// the global top kk).  Nothing in between reads a flag on the host: a query the coarse path cannot vouch for comes
// out of the merge with count -1 on EVERY rank and the caller redoes it with the exact kernels.
static bool batch_plan_global(svsb_engine* e, const Generation* g, int32_t k, BatchPlan& P) {
    if (!batch_plan(e, g, k, P)) return false;
    // sample fraction f with kk * f ~ 3: the union's order statistic of rank ~ 3 + 6 sqrt(3) + 4 < SAMPLE_TOPX
    // ... but no more than ONE wave of the sample pass (40 tiles x 4 query blocks of a 1024-query batch): a bigger sample
    // costs more than the tighter threshold saves in re-scored rows (profiles/r02_c3_phases_n2.txt: 118 tiles = 73 us)
    int64_t want = std::min<int64_t>((int64_t)std::ceil(3.0 * (double)g->n / (double)std::max(1, k)), 40 * COARSE_TILE_ROWS);
    if (const char* v = getenv("SVSB_BATCH_GLOBAL_SAMPLE_ROWS")) want = atoll(v);
    int64_t st = std::min<int64_t>(std::max<int64_t>((want + COARSE_TILE_ROWS - 1) / COARSE_TILE_ROWS, 2), P.n_tiles);
    P.s_tiles = (int)st;
    P.tile_stride = std::max(1, P.n_tiles / P.s_tiles);
    P.sample_rows = (int64_t)P.s_tiles * COARSE_TILE_ROWS;
    P.sample_alloc_rows = std::max(P.sample_alloc_rows, P.sample_rows);
    P.sample_rank = 0;                                   // the caller's: it depends on every rank's sample fraction
    return P.sample_rows >= 8 * SAMPLE_TOPX;             // launch_sample_top: SAMPLE_TOPX threads with at least one vector each
}

extern "C" int svsb_batch_global_probe(svsb_t* e, int32_t k, int32_t* eligible, int64_t* sample_rows, int64_t* local_rows,
                                       float* max_row_norm) {
    if (!e || !eligible || !sample_rows || !local_rows || !max_row_norm) return fail(SVSB_E_INVALID, "svsb_batch_global_probe: NULL argument");
    *eligible = 0; *sample_rows = 0; *local_rows = 0; *max_row_norm = 1.f;
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    *local_rows = g->n_live;
    BatchPlan P;
    if (k < 1 || k > K_FAST_MAX || env_int("SVSB_BATCH_GLOBAL", 1) == 0 || g->n_live == 0 || !batch_plan_global(e, g.get(), k, P)) return SVSB_OK;
    *eligible = 1; *sample_rows = P.sample_rows; *max_row_norm = P.max_row_norm;
    return SVSB_OK;
}

// The arguments the caller chose for ALL ranks must cover this shard: max_row_norm at least its own (and safe for fp16
// operands), sample_rank at least its own statistical bound (or SAMPLE_TOPX, all a rank ships).  svsb_batch_sample_tops
// has no sample_rank yet and passes SAMPLE_TOPX; svsb_batch_global_records takes the norm svsb_batch_sample_tops checked.
static int batch_global_check(const BatchPlan& P, float max_row_norm, int32_t sample_rank, const char* who) {
    if (!(max_row_norm >= P.max_row_norm) || !(max_row_norm <= 8.1f))
        return fail(SVSB_E_INVALID, std::string(who) + ": max_row_norm below this shard's own, or unsafe for fp16 operands");
    const double lam = (double)P.kk * std::min(1.0, (double)P.sample_rows / (double)P.n);
    if ((double)sample_rank < std::ceil(lam + 6.0 * std::sqrt(lam) + 4.0) && sample_rank < SAMPLE_TOPX && env_int("SVSB_BATCH_GLOBAL_ANY_RANK", 0) == 0)
        return fail(SVSB_E_INVALID, std::string(who) + ": sample_rank below this shard's own bound");
    return SVSB_OK;
}

extern "C" int svsb_batch_sample_tops(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, float max_row_norm, float* d_tops) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (b < 1 || b > COARSE_MAX_BATCH || !d_Q || !d_tops) return fail(SVSB_E_INVALID, "svsb_batch_sample_tops: 1 <= b <= 2048, non-NULL buffers");
    BatchPlan P;
    if (!batch_plan_global(e, g.get(), k, P)) return fail(SVSB_E_STATE, "svsb_batch_sample_tops: this shard / k is not eligible (svsb_batch_global_probe)");
    int rc = batch_global_check(P, max_row_norm, SAMPLE_TOPX, "svsb_batch_sample_tops");
    if (rc != SVSB_OK) return rc;
    P.max_row_norm = max_row_norm;
    cudaStream_t st = (cudaStream_t)stream;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = nullptr;
    if ((rc = batch_acquire(e, g.get(), P, b, st, w)) != SVSB_OK) return rc;
    if ((rc = batch_sample(w, g.get(), P, d_Q, b, st)) != SVSB_OK) return rc;
    CU(launch_sample_top(st, w->sample, P.sample_rows, b, d_tops));
    w->global_gen = g->id; w->global_b = b; w->global_k = k;
    return SVSB_OK;
}

extern "C" int svsb_batch_global_records(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, const float* d_tops_all,
                                         int32_t world, int32_t sample_rank, int32_t rec_cap, int64_t* d_records) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (b < 1 || b > COARSE_MAX_BATCH || !d_Q || !d_tops_all || !d_records) return fail(SVSB_E_INVALID, "svsb_batch_global_records: 1 <= b <= 2048, non-NULL buffers");
    if (world < 1 || world > XCHG_MAX_RANKS || sample_rank < 1 || sample_rank > SAMPLE_TOPX)
        return fail(SVSB_E_INVALID, "svsb_batch_global_records: 1 <= world <= 16, 1 <= sample_rank <= 32");
    if (rec_cap < 1 || rec_cap > k) return fail(SVSB_E_INVALID, "svsb_batch_global_records: 1 <= rec_cap <= k");
    BatchPlan P;
    if (!batch_plan_global(e, g.get(), k, P)) return fail(SVSB_E_STATE, "svsb_batch_global_records: this shard / k is not eligible");
    cudaStream_t st = (cudaStream_t)stream;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = e->batch_ws.get();
    if (!w || w->global_gen != g->id || w->global_b != b || w->global_k != k)
        return fail(SVSB_E_STATE, "svsb_batch_global_records: no matching svsb_batch_sample_tops call precedes it");
    w->global_gen = 0;
    int rc = batch_global_check(P, P.max_row_norm, sample_rank, "svsb_batch_global_records");
    if (rc != SVSB_OK) return rc;
    CU(cudaSetDevice(w->dev));
    CU(launch_union_threshold(st, d_tops_all, (int64_t)b * SAMPLE_TOPX, world, b, sample_rank, w->eps, w->thr));
    return batch_filter_refine(w, g.get(), P, d_Q, b, st, RecordView{d_records, rec_cap}.refine_out(true), REFINE_PARTIAL | REFINE_DEFER);
}

// ---- the same batch protocol with BOTH exchanges fused into the kernels over NVLink peer memory (no collective) -------
// svsb_batch_peer = svsb_batch_sample_tops + all-gather + svsb_batch_global_records + all-gather + verifying merge, except
// that the two all-gathers do not exist: the order-statistic kernel stores this rank's sample maxima straight into every
// rank's batch window and the sort kernel of the refine does the same with the candidate records (BatchPush: peer
// stores, a last-block ticket, a system-scope release of the batch's sequence number); the consumers -- the union
// threshold kernel, the merge -- run behind a one-CTA kernel that acquires the `world` flags of its OWN window.  At 8
// GPUs the two NCCL all-gathers were 75-85 us of a 380 us batch (profiles/r02_c3_phases_n8.txt).
// Slot reuse: everything of a batch is on one stream per rank, so a rank can only push batch j+1's maxima after its own
// merge of batch j (immediate form) or j-1 (pipelined form, flags bit 0) has seen every peer's records of that batch, which
// those peers pushed after reading all its maxima: the immediate form would do with one slot, the pipelined form needs the two
// it has (tests/test_batch_window_protocol.py checks the interleavings).
static void bxchg_release(svsb_engine* e) {
    BXchg* x = e->bxchg.get();
    if (!x) return;
    cudaSetDevice(e->devs[0]);
    cudaDeviceSynchronize();
    x->maps.close();
    if (x->block) cudaFree(x->block);
    if (x->done) cudaFree(x->done);
    if (x->status) cudaFree(x->status);
    (void)cudaGetLastError();
    e->bxchg.reset();
}

extern "C" int svsb_bxchg_create(svsb_t* e, int32_t world, int32_t rank, int32_t rec_cap, void* handle_out) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    int rc = check_world_rank(e, world, rank, "svsb_bxchg_create");
    if (rc != SVSB_OK) return rc;
    if (rec_cap < 1 || rec_cap > 1024) return fail(SVSB_E_INVALID, "svsb_bxchg_create: 1 <= rec_cap <= 1024");
    bxchg_release(e);
    e->bxchg.reset(new BXchg());
    BXchg* x = e->bxchg.get();
    x->world = world; x->rank = rank; x->rec_cap = rec_cap;
    x->flags_bytes = ((size_t)2 * BXchg::SLOTS * world * 8 + 255) & ~(size_t)255;
    x->tops_bytes = (size_t)BXchg::SLOTS * world * x->tops_region() * 4;
    x->bytes = x->flags_bytes + x->tops_bytes + (size_t)BXchg::SLOTS * world * x->rec_region() * 8;
    CU(cudaSetDevice(e->devs[0]));
    CU(preload_batch_kernels());             // lazy module loading synchronises the context at a kernel's first launch --
    CU(preload_coarse_kernels());            // while a wait kernel of another engine of this process may be spinning
    CU(preload_merge_kernels());
    CU(cudaMalloc(&x->block, x->bytes));
    CU(cudaMemset(x->block, 0, x->flags_bytes));
    CU(cudaMalloc(&x->done, 64)); CU(cudaMemset(x->done, 0, 64));
    CU(cudaMalloc(&x->status, 64)); CU(cudaMemset(x->status, 0, 64));
    CU(cudaDeviceSynchronize());
    return x->publish(handle_out);
}

extern "C" int svsb_bxchg_connect(svsb_t* e, const void* handles) {
    if (!e || !e->bxchg) return fail(SVSB_E_STATE, "svsb_bxchg_connect: svsb_bxchg_create first");
    if (!handles) return fail(SVSB_E_INVALID, "svsb_bxchg_connect: NULL handles");
    CU(cudaSetDevice(e->devs[0]));
    return e->bxchg->connect(handles, "svsb_bxchg_connect");
}

extern "C" int svsb_bxchg_connect_local(svsb_t* e, svsb_t* const* engines) {
    if (!e || !e->bxchg) return fail(SVSB_E_STATE, "svsb_bxchg_connect_local: svsb_bxchg_create first");
    if (!engines) return fail(SVSB_E_INVALID, "svsb_bxchg_connect_local: NULL engines");
    CU(cudaSetDevice(e->devs[0]));
    return e->bxchg->connect_local(e->devs[0], engines, [](svsb_engine* o, const PeerWindow* self) -> PeerWindow* {
        return o->bxchg && o->bxchg->rec_cap == static_cast<const BXchg*>(self)->rec_cap ? o->bxchg.get() : nullptr;
    }, "svsb_bxchg_connect_local");
}

// Stop pushing into the peers' windows (they may be freed next); the own window stays until svsb_destroy / the next create.
extern "C" int svsb_bxchg_disconnect(svsb_t* e) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    BXchg* x = e->bxchg.get();
    if (!x) return SVSB_OK;
    CU(cudaSetDevice(e->devs[0]));
    CU(cudaDeviceSynchronize());
    x->unmap();
    x->deferred.pending = false;             // a merge nobody flushed dies with the connection
    return SVSB_OK;
}

// Size every buffer svsb_batch_peer uses for (b, k) now: allocations are implicit synchronisation points, and several
// shard engines of ONE process (tests with virtual ranks) must not hit one while another engine's wait kernel spins.
extern "C" int svsb_batch_peer_prepare(svsb_t* e, int32_t b, int32_t k) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (b < 1 || b > COARSE_MAX_BATCH) return fail(SVSB_E_INVALID, "svsb_batch_peer_prepare: 1 <= b <= 2048");
    BatchPlan P;
    if (!batch_plan_global(e, g.get(), k, P)) return fail(SVSB_E_STATE, "svsb_batch_peer_prepare: this shard / k is not eligible (svsb_batch_global_probe)");
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = nullptr;
    int rc = batch_acquire(e, g.get(), P, b, nullptr, w);
    if (rc != SVSB_OK) return rc;
    CU(cudaSetDevice(w->dev));
    CU(cudaDeviceSynchronize());
    return SVSB_OK;
}

// wait for every rank's records of the deferred batch, then the verifying merge
static int bxchg_enqueue_merge(svsb_engine* e, cudaStream_t st, const BXchg::Deferred& d) {
    BXchg* x = e->bxchg.get();
    CU(launch_wait_flags(st, x->flag(x->block, 1, d.slot, 0), x->world, d.seq, x->timeout_ns, x->status));
    return engine_merge_records(e, st, RecordView{x->recs(x->block, d.slot, 0), d.rec_cap}, x->world, x->rec_region(), d.b, d.k,
                                d.out_scores, d.out_ids, d.out_counts, d.k, x->status);
}

extern "C" int svsb_batch_peer_flush(svsb_t* e, void* stream) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    BXchg* x = e->bxchg.get();
    if (!x || !x->deferred.pending) return SVSB_OK;
    CU(cudaSetDevice(e->devs[0]));
    std::lock_guard<std::mutex> lk(e->batch_mu);
    int rc = bxchg_enqueue_merge(e, (cudaStream_t)stream, x->deferred);
    x->deferred.pending = false;
    return rc;
}

extern "C" int svsb_batch_peer(svsb_t* e, void* stream, const float* d_Q, int32_t b, int32_t k, float max_row_norm, int32_t sample_rank,
                               int32_t rec_cap, float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_counts, int32_t flags) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    BXchg* x = e->bxchg.get();
    if (!x || !x->connected) return fail(SVSB_E_STATE, "svsb_batch_peer: svsb_bxchg_create + svsb_bxchg_connect first");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (b < 1 || b > COARSE_MAX_BATCH || !d_Q || !d_out_scores || !d_out_ids || !d_out_counts)
        return fail(SVSB_E_INVALID, "svsb_batch_peer: 1 <= b <= 2048, non-NULL buffers");
    if (sample_rank < 1 || sample_rank > SAMPLE_TOPX) return fail(SVSB_E_INVALID, "svsb_batch_peer: 1 <= sample_rank <= 32");
    if (rec_cap < 1 || rec_cap > k || rec_cap > x->rec_cap) return fail(SVSB_E_INVALID, "svsb_batch_peer: rec_cap must be <= k and <= the window's");
    if (rec_cap < k && (int64_t)x->world * rec_cap > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_batch_peer: truncated records need world * rec_cap <= 2048");
    BatchPlan P;
    if (!batch_plan_global(e, g.get(), k, P)) return fail(SVSB_E_STATE, "svsb_batch_peer: this shard / k is not eligible (svsb_batch_global_probe)");
    int rc = batch_global_check(P, max_row_norm, sample_rank, "svsb_batch_peer");
    if (rc != SVSB_OK) return rc;
    P.max_row_norm = max_row_norm;
    cudaStream_t st = (cudaStream_t)stream;
    std::lock_guard<std::mutex> lk(e->batch_mu);
    BatchWs* w = nullptr;
    if ((rc = batch_acquire(e, g.get(), P, b, st, w)) != SVSB_OK) return rc;
    const unsigned long long seq = ++x->seq;
    const int slot = (int)(seq % BXchg::SLOTS);
    BatchPush pa, pb;
    pa.world = pb.world = x->world; pa.seq = pb.seq = seq; pa.done = x->done; pb.done = x->done + 1;
    for (int p = 0; p < x->world; ++p) {
        pa.dst[p] = x->tops(x->peer_block[p], slot, x->rank); pa.flag[p] = x->flag(x->peer_block[p], 0, slot, x->rank);
        pb.dst[p] = x->recs(x->peer_block[p], slot, x->rank); pb.flag[p] = x->flag(x->peer_block[p], 1, slot, x->rank);
    }
    // 1. this rank's sample maxima -> every rank's window
    if ((rc = batch_sample(w, g.get(), P, d_Q, b, st)) != SVSB_OK) return rc;
    CU(launch_sample_top(st, w->sample, P.sample_rows, b, nullptr, &pa));
    if (x->deferred.pending) {                 // the previous batch's merge: its peers had this phase's time to deliver
        rc = bxchg_enqueue_merge(e, st, x->deferred);
        x->deferred.pending = false;
        if (rc != SVSB_OK) return rc;
    }
    // 2. all ranks' maxima are here -> ONE threshold per query; filter; exact re-score; records -> every rank's window
    CU(launch_wait_flags(st, x->flag(x->block, 0, slot, 0), x->world, seq, x->timeout_ns, x->status));
    CU(launch_union_threshold(st, x->tops(x->block, slot, 0), x->tops_region(), x->world, b, sample_rank, w->eps, w->thr));
    if ((rc = batch_filter_refine(w, g.get(), P, d_Q, b, st, RecordView{nullptr, rec_cap}.refine_out(true), REFINE_PARTIAL | REFINE_DEFER, &pb)) != SVSB_OK)
        return rc;
    // 3. all ranks' records are here -> verifying merge (now, or behind the first phase of the next batch)
    BXchg::Deferred d;
    d.pending = true; d.slot = slot; d.rec_cap = rec_cap; d.k = k; d.b = b; d.seq = seq;
    d.out_scores = d_out_scores; d.out_ids = d_out_ids; d.out_counts = d_out_counts;
    if (flags & 1) { x->deferred = d; return SVSB_OK; }
    return bxchg_enqueue_merge(e, st, d);
}

// ---- peer exchange: the fused selection + exchange step and the waiting merge (kernels.cuh, select.cu) -------------
static int xchg_prepare(svsb_engine* e, const Generation* g);
static int xchg_flush_merge(svsb_engine* e, cudaStream_t st_sel);
extern "C" int svsb_xchg_create(svsb_t* e, int32_t world, int32_t rank, int32_t k_max, void* handle_out) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    int rc = check_world_rank(e, world, rank, "svsb_xchg_create");
    if (rc != SVSB_OK) return rc;
    if (k_max < 1 || k_max > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_xchg_create: 1 <= k_max <= 2048");
    xchg_release(e);
    e->xchg.reset(new Xchg());                 // owned by the engine from the start: a failure below leaves a window that
    Xchg* x = e->xchg.get();                   // is not `connected`; the next create / svsb_destroy releases what exists
    x->world = world; x->rank = rank; x->cap = k_max; x->rec_words = 2 * (int64_t)k_max + 2;
    x->flags_bytes = ((size_t)x->slots * world * 8 + 255) & ~(size_t)255;
    const size_t bytes = x->flags_bytes + (size_t)x->slots * world * x->rec_words * 8;
    CU(cudaSetDevice(e->devs[0]));
    CU(preload_gemv_kernels());
    CU(preload_peer_kernels());
    CU(cudaMalloc(&x->block, bytes));
    CU(cudaMemset(x->block, 0, bytes));
    CU(cudaDeviceSynchronize());
    CU(cudaStreamCreateWithFlags(&x->st, cudaStreamNonBlocking));
    x->ws.dev = e->devs[0]; x->ws.st = x->st;
    CU(cudaMallocHost(&x->h_scores, (size_t)k_max * 4));
    CU(cudaMallocHost(&x->h_ids, (size_t)k_max * 8));
    CU(cudaMallocHost(&x->h_count, 64));
    x->h_cap = k_max;
    if (env_int("SVSB_XCHG_STAMPS", 0)) {
        CU(cudaMalloc(&x->stamps, (size_t)Xchg::STAMP_RING * Xchg::STAMP_WORDS * 8));
        CU(cudaMemset(x->stamps, 0, (size_t)Xchg::STAMP_RING * Xchg::STAMP_WORDS * 8));
        CU(cudaDeviceSynchronize());
    }
    return x->publish(handle_out);
}

// Close the peers' windows (this rank stops pushing) but keep the own one alive: peers may still have it mapped.
// Shutdown order across ranks: disconnect everywhere, barrier, then svsb_destroy.
extern "C" int svsb_xchg_disconnect(svsb_t* e) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    Xchg* x = e->xchg.get();
    if (!x) return SVSB_OK;
    CU(cudaSetDevice(e->devs[0]));
    if (x->deferred.pending && e->side_st) { int rc = xchg_flush_merge(e, e->side_st); if (rc != SVSB_OK) return rc; }
    if (x->st) CU(cudaStreamSynchronize(x->st));
    if (e->side_st) CU(cudaStreamSynchronize(e->side_st));
    x->unmap();
    return SVSB_OK;
}

extern "C" int svsb_xchg_connect(svsb_t* e, const void* handles) {
    if (!e || !e->xchg) return fail(SVSB_E_STATE, "svsb_xchg_connect: svsb_xchg_create first");
    if (!handles) return fail(SVSB_E_INVALID, "svsb_xchg_connect: NULL handles");
    CU(cudaSetDevice(e->devs[0]));
    int rc = e->xchg->connect(handles, "svsb_xchg_connect");
    if (rc != SVSB_OK) return rc;
    if (auto g = pin(e)) return xchg_prepare(e, g.get());
    return SVSB_OK;
}

extern "C" int svsb_xchg_connect_local(svsb_t* e, svsb_t* const* engines) {
    if (!e || !e->xchg) return fail(SVSB_E_STATE, "svsb_xchg_connect_local: svsb_xchg_create first");
    if (!engines) return fail(SVSB_E_INVALID, "svsb_xchg_connect_local: NULL engines");
    CU(cudaSetDevice(e->devs[0]));
    int rc = e->xchg->connect_local(e->devs[0], engines, [](svsb_engine* o, const PeerWindow* self) -> PeerWindow* {
        return o->xchg && o->xchg->cap == static_cast<const Xchg*>(self)->cap ? o->xchg.get() : nullptr;
    }, "svsb_xchg_connect_local");
    if (rc != SVSB_OK) return rc;
    if (auto g = pin(e)) return xchg_prepare(e, g.get());
    return SVSB_OK;
}

// Size every buffer the peer paths use for the resident generation.  Allocations, memsets and pinned allocations are
// implicit synchronisation points of the CUDA runtime: issued while another engine OF THIS PROCESS has a merge kernel
// spinning on a flag they can deadlock, so they all happen here -- at connect time and (a no-op once sized) at the
// top of each call, before anything of that call is enqueued.
static int xchg_prepare(svsb_engine* e, const Generation* g) {
    Xchg* x = e->xchg.get();
    const Shard& s = g->shards[0];
    CU(cudaSetDevice(s.dev));
    if (!e->side_st) CU(cudaStreamCreateWithFlags(&e->side_st, cudaStreamNonBlocking));
    int rc;
    for (DevWs* w : {&x->ws, &shard_slot(e, 0), &shard_slot(e, 1)}) {
        if ((rc = w->ensure_set(s.n)) != SVSB_OK) return rc;
        if ((int64_t)x->world * x->cap > K_FAST_MAX && (rc = w->ensure_merge_scratch((int64_t)x->world * x->cap)) != SVSB_OK) return rc;
    }
    if ((rc = x->ws.ensure_q(g->ld)) != SVSB_OK) return rc;
    if (g->ld > x->h_q_cap) {
        if (x->h_q) cudaFreeHost(x->h_q);
        x->h_q = nullptr; x->h_q_cap = 0;
        CU(cudaMallocHost(&x->h_q, (size_t)g->ld * 4));
        x->h_q_cap = g->ld;
    }
    cudaEvent_t* t;                                              // the timing bracket of the call's pass, if it asks
    if ((rc = kev_next(e, t)) != SVSB_OK) return rc;
    if (!x->ev_join) CU(cudaEventCreateWithFlags(&x->ev_join, cudaEventDisableTiming));
    return SVSB_OK;
}

// Fill the push descriptor for the next query and return its window slot.
static int xchg_next(Xchg* x, PeerPush& push) {
    const unsigned long long seq = ++x->seq;
    const int slot = (int)(seq % (unsigned long long)x->slots);
    push.world = x->world; push.cap = x->cap; push.seq = seq;
    for (int p = 0; p < x->world; ++p) {
        push.rec[p] = x->rec_of(x->peer_block[p], slot, x->rank);
        push.flag[p] = x->flags_of(x->peer_block[p], slot) + x->rank;
    }
    return slot;
}

static int xchg_flush_merge(svsb_engine* e, cudaStream_t st_sel) {
    Xchg* x = e->xchg.get();
    Xchg::DeferredMerge& m = x->deferred;
    if (!m.pending) return SVSB_OK;
    m.pending = false;
    CU(launch_merge_window(st_sel, x->rec_of(x->block, m.slot, 0), x->flags_of(x->block, m.slot), m.seq, x->world, x->cap, m.k,
                           x->timeout_ns, m.sk, m.sp, m.out_scores, m.out_ids, m.out_count));
    if (m.ev_done) { CU(cudaEventRecord(m.ev_done, st_sel)); m.ev_done = nullptr; }
    return SVSB_OK;
}

// similarity on st_main, then (on st_sel) selection with the fused push and the waiting merge into out_*.
// pipelined: ev_sel marks the end of the selection (scores reusable by the similarity pass two queries on), and the merge
// is enqueued by the NEXT call (or by svsb_enqueue_join), behind that call's selection.
// Window slots stay safe with 4 of them: a rank pushes query j+4 after its merge(j+2), i.e. after every peer pushed
// j+2, and each peer enqueues merge(j) before its selection j+2.
static int xchg_enqueue(svsb_engine* e, const Generation* g, DevWs& w, cudaStream_t st_main, cudaStream_t st_sel,
                        const float* d_query, int32_t k, float* out_scores, int64_t* out_ids, int32_t* out_count,
                        bool time_kernel, int reserve_sms, bool pipelined, bool pdl_gemv = false) {
    Xchg* x = e->xchg.get();
    const Shard& s = g->shards[0];
    PeerPush push{};
    const int slot = xchg_next(x, push);
    int rc;
    if (s.n_live == 0) {
        CU(launch_push_empty(st_sel, push));
    } else {
        cudaEvent_t* t = nullptr;
        if (time_kernel && (rc = kev_next(e, t)) != SVSB_OK) return rc;
        // route 0 on purpose, as in enqueue_local_topk_gen; PDL only after the staging kernel of the host-buffer paths
        if ((rc = similarity_phase(st_main, w, g, s, d_query, 0, reserve_sms, pdl_gemv, t)) != SVSB_OK) return rc;
        if (t) e->kev_used += 2;
        if (st_sel != st_main && (rc = w.hand_off(st_main, st_sel)) != SVSB_OK) return rc;
        u64* sel_stamps = (x->stamps && !pipelined) ? x->stamps + (push.seq % Xchg::STAMP_RING) * Xchg::STAMP_WORDS : nullptr;
        if ((rc = select_phase(st_sel, w, g, s, d_query, 0, k, w.out(), sel_stamps, &push)) != SVSB_OK) return rc;
    }
    if (pipelined) { CU(cudaEventRecord(w.ev_sel, st_sel)); w.sel_pending = true; }
    u64* sk = nullptr; int64_t* sp = nullptr;
    if ((int64_t)x->world * k > K_FAST_MAX) { sk = w.mscr_keys; sp = w.mscr_ids; }
    if (pipelined) {
        if ((rc = xchg_flush_merge(e, st_sel)) != SVSB_OK) return rc;   // the previous query's merge goes behind this selection
        Xchg::DeferredMerge& m = x->deferred;
        m.pending = true; m.slot = slot; m.k = k; m.seq = push.seq; m.sk = sk; m.sp = sp;
        m.out_scores = out_scores; m.out_ids = out_ids; m.out_count = out_count; m.ev_done = nullptr;
        return SVSB_OK;
    }
    CU(launch_merge_window(st_sel, x->rec_of(x->block, slot, 0), x->flags_of(x->block, slot), push.seq, x->world, x->cap, k,
                           x->timeout_ns, sk, sp, out_scores, out_ids, out_count,
                           x->stamps ? x->stamps + (push.seq % Xchg::STAMP_RING) * Xchg::STAMP_WORDS + 16 : nullptr));
    return SVSB_OK;
}

extern "C" int svsb_enqueue_query_peer(svsb_t* e, void* stream, const float* d_query, int32_t k,
                                       float* out_scores, int64_t* out_ids, int32_t* out_count, int32_t flags) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!e->xchg || !e->xchg->connected) return fail(SVSB_E_STATE, "svsb_enqueue_query_peer: exchange not connected");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (k < 1 || k > e->xchg->cap) return fail(SVSB_E_INVALID, "svsb_enqueue_query_peer: 1 <= k <= k_max of the exchange");
    if (!d_query || !out_scores || !out_ids || !out_count) return fail(SVSB_E_INVALID, "svsb_enqueue_query_peer: NULL pointer");
    const bool time_kernel = (flags & 1) != 0, pipelined = (flags & 2) != 0;
    const Shard& s = g->shards[0];
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaSetDevice(s.dev));
    int rc = xchg_prepare(e, g.get());
    if (rc != SVSB_OK) return rc;
    const int slot = (int)(e->xchg->seq & 1);              // workspace set: alternates so that query i+1's similarity pass
    DevWs& w = shard_slot(e, slot);                        // overlaps query i's selection
    if (!pipelined && e->xchg->deferred.pending && (rc = xchg_flush_merge(e, e->side_st)) != SVSB_OK) return rc;
    // the set's scores are free again (a plain call after a pipelined one on this set, too)
    if ((rc = w.sel_wait(st)) != SVSB_OK) return rc;
    if (!pipelined) w.sel_pending = false;
    return xchg_enqueue(e, g.get(), w, st, pipelined ? e->side_st : st, d_query, k, out_scores, out_ids, out_count, time_kernel,
                        pipelined ? 1 : 0, pipelined);
}

extern "C" int svsb_query_peer(svsb_t* e, const float* q, int32_t d, int32_t k,
                               float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!out_count) return fail(SVSB_E_INVALID, "svsb_query_peer: out_count is NULL");
    *out_count = 0;
    if (!e->xchg || !e->xchg->connected) return fail(SVSB_E_STATE, "svsb_query_peer: exchange not connected");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (d != g->d) return fail(SVSB_E_SHAPE, "svsb_query_peer: query dimension does not match the matrix");
    Xchg* x = e->xchg.get();
    if (k < 1 || k > x->cap) return fail(SVSB_E_INVALID, "svsb_query_peer: 1 <= k <= k_max of the exchange");
    if (!q || !out_scores || !out_emb_ids) return fail(SVSB_E_INVALID, "svsb_query_peer: NULL buffer");
    int rc = xchg_prepare(e, g.get());
    if (rc != SVSB_OK) return rc;
    if (x->deferred.pending && (rc = xchg_flush_merge(e, e->side_st)) != SVSB_OK) return rc;   // keep merges in sequence order
    stage_queries(x->h_q, q, 1, d, g->ld);
    CU(launch_stage_query(x->st, x->h_q, x->ws.d_q, g->ld));     // a kernel reads the pinned query: no copy-engine hop
    *x->h_count = -1;
    // the merge kernel writes the result into pinned (mapped) host memory: no copy back, one synchronize
    if ((rc = xchg_enqueue(e, g.get(), x->ws, x->st, x->st, x->ws.d_q, k, x->h_scores, x->h_ids, x->h_count, false, 0,
                           /*pipelined=*/false, /*pdl_gemv=*/env_int("SVSB_PDL", 1) != 0)) != SVSB_OK) return rc;
    CU(cudaStreamSynchronize(x->st));
    const int32_t cnt = *x->h_count;
    if (cnt == MERGE_WINDOW_TIMED_OUT)
        return fail(SVSB_E_STATE, "svsb_query_peer: a peer's record did not arrive in time (a rank died or left the call sequence)");
    if (cnt < 0 || cnt > k) return fail(SVSB_E_CUDA, "svsb_query_peer: internal: merge returned a bad count");
    memcpy(out_scores, x->h_scores, (size_t)cnt * 4);
    memcpy(out_emb_ids, x->h_ids, (size_t)cnt * 8);
    *out_count = cnt;
    return SVSB_OK;
}

// ---- the synchronous peer query with several in flight: submit / wait ---------------------------------------------
// Same kernels as svsb_query_peer, arranged like the device-resident pipelined loop: the similarity pass runs on the
// exchange's stream leaving one SM free, selection + push and the (deferred) waiting merge run on the side stream, so
// query j+1's matrix pass overlaps query j's selection, exchange, merge and host round trip.
static int xchg_ensure_tickets(svsb_engine* e, const Generation* g) {
    Xchg* x = e->xchg.get();
    CU(cudaSetDevice(e->devs[0]));
    const bool grow = g->ld > x->tk_ld;
    for (auto& t : x->tk) {
        if (t.busy && grow) return fail(SVSB_E_STATE, "svsb_query_peer_submit: the matrix changed shape with queries pending");
        if (grow) {
            if (t.h_q) cudaFreeHost(t.h_q);
            if (t.d_q) cudaFree(t.d_q);
            t.h_q = nullptr; t.d_q = nullptr;
            CU(cudaMallocHost(&t.h_q, (size_t)g->ld * 4));
            CU(cudaMalloc(&t.d_q, (size_t)g->ld * 4));
        }
        if (!t.h_scores) {
            CU(cudaMallocHost(&t.h_scores, (size_t)x->cap * 4));
            CU(cudaMallocHost(&t.h_ids, (size_t)x->cap * 8));
            CU(cudaMallocHost(&t.h_count, 64));
            CU(cudaEventCreateWithFlags(&t.ev, cudaEventDisableTiming));
        }
    }
    if (grow) x->tk_ld = g->ld;
    return SVSB_OK;
}

extern "C" int svsb_query_peer_submit(svsb_t* e, const float* q, int32_t d, int32_t k, int32_t* ticket) {
    if (!e || !ticket) return fail(SVSB_E_INVALID, "svsb_query_peer_submit: NULL argument");
    *ticket = -1;
    if (!e->xchg || !e->xchg->connected) return fail(SVSB_E_STATE, "svsb_query_peer_submit: exchange not connected");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (d != g->d) return fail(SVSB_E_SHAPE, "svsb_query_peer_submit: query dimension does not match the matrix");
    Xchg* x = e->xchg.get();
    if (k < 1 || k > x->cap) return fail(SVSB_E_INVALID, "svsb_query_peer_submit: 1 <= k <= k_max of the exchange");
    if (!q) return fail(SVSB_E_INVALID, "svsb_query_peer_submit: NULL buffer");
    int rc = xchg_prepare(e, g.get());
    if (rc != SVSB_OK) return rc;
    if ((rc = xchg_ensure_tickets(e, g.get())) != SVSB_OK) return rc;
    const int ti = x->tk_next;
    Xchg::Ticket& t = x->tk[ti];
    if (t.busy) return fail(SVSB_E_STATE, "svsb_query_peer_submit: 3 queries are pending already (wait for the oldest first)");
    stage_queries(t.h_q, q, 1, d, g->ld);
    *t.h_count = -1;
    DevWs& w = shard_slot(e, x->seq & 1);                      // workspace set (xchg_enqueue takes sequence number seq + 1)
    CU(cudaSetDevice(e->devs[0]));
    if ((rc = w.sel_wait(x->st)) != SVSB_OK) return rc;        // the set's previous selection is done with it
    CU(launch_stage_query(x->st, t.h_q, t.d_q, g->ld));
    rc = xchg_enqueue(e, g.get(), w, x->st, e->side_st, t.d_q, k, t.h_scores, t.h_ids, t.h_count, false, /*reserve_sms=*/1,
                      /*pipelined=*/true, /*pdl_gemv=*/env_int("SVSB_PDL", 1) != 0);
    if (rc != SVSB_OK) return rc;
    x->deferred.ev_done = t.ev;                                // recorded when this query's merge is enqueued
    t.busy = true; t.k = k; t.seq = x->seq;
    x->tk_next = (ti + 1) % Xchg::N_TICKETS;
    *ticket = ti;
    return SVSB_OK;
}

extern "C" int svsb_query_peer_wait(svsb_t* e, int32_t ticket, float* out_scores, int64_t* out_emb_ids, int32_t* out_count) {
    if (!e || !out_count) return fail(SVSB_E_INVALID, "svsb_query_peer_wait: NULL argument");
    *out_count = 0;
    if (!e->xchg) return fail(SVSB_E_STATE, "svsb_query_peer_wait: no exchange");
    Xchg* x = e->xchg.get();
    if (ticket < 0 || ticket >= Xchg::N_TICKETS || !x->tk[ticket].busy) return fail(SVSB_E_INVALID, "svsb_query_peer_wait: no such pending query");
    Xchg::Ticket& t = x->tk[ticket];
    CU(cudaSetDevice(e->devs[0]));
    if (x->deferred.pending && x->deferred.seq == t.seq) {      // nobody submitted behind it: enqueue its merge now
        int rc = xchg_flush_merge(e, e->side_st);
        if (rc != SVSB_OK) { t.busy = false; return rc; }
    }
    t.busy = false;
    CU(cudaEventSynchronize(t.ev));
    const int32_t cnt = *t.h_count;
    if (cnt == MERGE_WINDOW_TIMED_OUT)
        return fail(SVSB_E_STATE, "svsb_query_peer_wait: a peer's record did not arrive in time (a rank died or left the call sequence)");
    if (cnt < 0 || cnt > t.k) return fail(SVSB_E_CUDA, "svsb_query_peer_wait: internal: merge returned a bad count");
    if (cnt > 0 && (!out_scores || !out_emb_ids)) return fail(SVSB_E_INVALID, "svsb_query_peer_wait: NULL buffer");
    memcpy(out_scores, t.h_scores, (size_t)cnt * 4);
    memcpy(out_emb_ids, t.h_ids, (size_t)cnt * 8);
    *out_count = cnt;
    return SVSB_OK;
}

// Measurement aid: copy the stamp ring (SVSB_XCHG_STAMPS=1 at svsb_xchg_create) to the host: STAMP_RING x 40 u64, entry
// seq % 1024 = [16 selection-kernel stamps (svsb_debug_select_phases layout) | seq, merge start, merge done, -, flag seen x world].
extern "C" int svsb_xchg_read_stamps(svsb_t* e, uint64_t* out, int64_t capacity_words) {
    if (!e || !out) return fail(SVSB_E_INVALID, "svsb_xchg_read_stamps: NULL argument");
    if (!e->xchg || !e->xchg->stamps) return fail(SVSB_E_STATE, "svsb_xchg_read_stamps: create the exchange with SVSB_XCHG_STAMPS=1");
    const int64_t words = (int64_t)Xchg::STAMP_RING * Xchg::STAMP_WORDS;
    if (capacity_words < words) return fail(SVSB_E_INVALID, "svsb_xchg_read_stamps: buffer too small (1024 x 40 words)");
    CU(cudaSetDevice(e->devs[0]));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out, e->xchg->stamps, (size_t)words * 8, cudaMemcpyDeviceToHost));
    return SVSB_OK;
}

extern "C" int svsb_enqueue_join(svsb_t* e, void* stream) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    CU(cudaSetDevice(e->devs[0]));
    if (e->xchg && e->xchg->deferred.pending && e->side_st) {       // the last peer query's merge, then everything on the side stream
        int rc = xchg_flush_merge(e, e->side_st);
        if (rc != SVSB_OK) return rc;
    }
    if (e->xchg && e->xchg->ev_join && e->side_st) {
        CU(cudaEventRecord(e->xchg->ev_join, e->side_st));
        CU(cudaStreamWaitEvent((cudaStream_t)stream, e->xchg->ev_join, 0));
    }
    for (auto& w : e->shard_ws) {
        int rc;
        if (w && (rc = w->sel_wait((cudaStream_t)stream)) != SVSB_OK) return rc;
    }
    return SVSB_OK;
}

extern "C" int svsb_kernel_time_collect(svsb_t* e, float* ms) {
    if (!e || !ms) return fail(SVSB_E_INVALID, "svsb_kernel_time_collect: NULL argument");
    float sum = 0.f;
    CU(cudaSetDevice(e->devs[0]));
    for (size_t i = 0; i + 1 < e->kev_used; i += 2) {
        CU(cudaEventSynchronize(e->kev[i + 1]));
        float t = 0.f; CU(cudaEventElapsedTime(&t, e->kev[i], e->kev[i + 1])); sum += t;
    }
    e->kev_used = 0;
    *ms = sum;
    return SVSB_OK;
}

static int enqueue_merge_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t batch, int32_t cap,
                                 int32_t k, float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_counts, int verify_k, const char* who) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (n_lists < 1 || batch < 1 || k < 1 || k > K_FAST_MAX || cap < 1 || cap > k) return fail(SVSB_E_INVALID, std::string(who) + ": bad arguments");
    if (cap < k && ((int64_t)n_lists * cap > K_FAST_MAX || n_lists > 16)) return fail(SVSB_E_INVALID, std::string(who) + ": truncated records need n_lists <= 16 and n_lists * rec_cap <= 2048");
    if (!d_records || !d_out_scores || !d_out_ids || !d_out_counts) return fail(SVSB_E_INVALID, std::string(who) + ": NULL pointer");
    CU(cudaSetDevice(e->devs[0]));
    const RecordView recs{const_cast<int64_t*>(d_records), cap};           // read only
    return engine_merge_records(e, (cudaStream_t)stream, recs, n_lists, (int64_t)batch * recs.words(), batch, k,
                                d_out_scores, d_out_ids, d_out_counts, verify_k);
}
extern "C" int svsb_enqueue_merge_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t batch,
                                          int32_t k, float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_counts) {
    return enqueue_merge_records(e, stream, d_records, n_lists, batch, k, k, d_out_scores, d_out_ids, d_out_counts, -1, "svsb_enqueue_merge_records");
}
extern "C" int svsb_enqueue_merge_sorted_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t cap,
                                                 int32_t k, float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_count) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (n_lists < 1 || cap < 1 || k < 1) return fail(SVSB_E_INVALID, "svsb_enqueue_merge_sorted_records: n_lists, cap and k must be positive");
    if (!d_records || !d_out_scores || !d_out_ids || !d_out_count)
        return fail(SVSB_E_INVALID, "svsb_enqueue_merge_sorted_records: NULL pointer");
    CU(cudaSetDevice(e->devs[0]));
    const RecordView recs{const_cast<int64_t*>(d_records), cap};           // read only
    CU(launch_merge_sorted_big((cudaStream_t)stream, recs.keys(0), recs.ids(0), recs.count(0), n_lists, cap, recs.words(),
                               2 * recs.words(), k, d_out_scores, d_out_ids, d_out_count));
    return SVSB_OK;
}
extern "C" int svsb_enqueue_merge_batch_records(svsb_t* e, void* stream, const int64_t* d_records, int32_t n_lists, int32_t batch,
                                                int32_t rec_cap, int32_t k, int32_t verify_k, float* d_out_scores, int64_t* d_out_ids,
                                                int32_t* d_out_counts) {
    if (verify_k < 0 || verify_k > k) return fail(SVSB_E_INVALID, "svsb_enqueue_merge_batch_records: 0 <= verify_k <= k");
    return enqueue_merge_records(e, stream, d_records, n_lists, batch, rec_cap, k, d_out_scores, d_out_ids, d_out_counts, verify_k, "svsb_enqueue_merge_batch_records");
}

// ------------------------------------------------------------------------------------------------
// stateless launchers (one process per GPU; torch owns memory and streams)
// ------------------------------------------------------------------------------------------------
extern "C" int svsb_ws_create(int device, int64_t n_rows, int32_t k_max, svsb_ws_t** out) {
    if (!out) return fail(SVSB_E_INVALID, "svsb_ws_create: out is NULL");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) {
        (void)cudaGetLastError();
        return fail(SVSB_E_NO_DEVICE, "svsb_ws_create: no such CUDA device; svs_b200 has no CPU path");
    }
    if (n_rows < 0 || n_rows > 0xfffffff0ll) return fail(SVSB_E_INVALID, "svsb_ws_create: bad n_rows");
    std::unique_ptr<svsb_workspace> w(new svsb_workspace());
    w->dev = device;
    int rc;
    // n_rows = 0: outputs only (rows and the sort buffer are sized by the first launch)
    if ((rc = w->ensure_query(n_rows, std::max<int64_t>(k_max, 128), n_rows > 0 ? k_max : 0)) != SVSB_OK) { w->release(); return rc; }
    *out = w.release();
    return SVSB_OK;
}

extern "C" void svsb_ws_destroy(svsb_ws_t* ws) {
    if (!ws) return;
    ws->release();
    delete ws;
}

extern "C" int svsb_launch_local_topk(svsb_ws_t* ws, void* stream, const float* d_matrix, int64_t n, int32_t d,
                                      int32_t ld, const int64_t* d_emb_ids, int64_t global_row0, const float* d_query,
                                      int32_t k, uint64_t* d_out_keys, int64_t* d_out_ids, int32_t* d_out_count) {
    if (!ws) return fail(SVSB_E_INVALID, "workspace is NULL");
    if (n <= 0 || d <= 0 || ld < d || (ld & 3)) return fail(SVSB_E_INVALID, "svsb_launch_local_topk: bad shape (ld must be a multiple of 4, >= d)");
    if (k <= 0) return fail(SVSB_E_INVALID, "svsb_launch_local_topk: k must be positive");
    if (!d_matrix || !d_query || !d_out_keys || !d_out_ids || !d_out_count) return fail(SVSB_E_INVALID, "svsb_launch_local_topk: NULL pointer");
    const int64_t kk = std::min<int64_t>(k, n);
    int rc;
    if ((rc = ws->ensure_query(n, std::max<int64_t>(kk, 128), kk)) != SVSB_OK) return rc;
    CU(cudaSetDevice(ws->dev));
    // the caller's rows as a shard of one generation; they are only read
    Generation g; g.d = d; g.ld = ld;
    Shard s; s.dev = ws->dev; s.row0 = global_row0; s.n = s.n_live = n;
    s.M = const_cast<float*>(d_matrix); s.ids = const_cast<int64_t*>(d_emb_ids);
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = similarity_phase(st, *ws, &g, s, d_query, 0)) != SVSB_OK) return rc;
    return select_phase(st, *ws, &g, s, d_query, 0, kk, {(u64*)d_out_keys, ws->out_scores, d_out_ids, d_out_count});
}

extern "C" int svsb_launch_merge(svsb_ws_t* ws, void* stream, const uint64_t* d_keys, const int64_t* d_ids,
                                 const int32_t* d_counts, int32_t n_lists, int32_t stride, int32_t k,
                                 float* d_out_scores, int64_t* d_out_ids, int32_t* d_out_count) {
    if (!ws) return fail(SVSB_E_INVALID, "workspace is NULL");
    if (n_lists < 1 || stride < 1 || k < 1 || k > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_launch_merge: bad arguments (k <= 2048)");
    if (!d_keys || !d_ids || !d_counts || !d_out_scores || !d_out_ids || !d_out_count) return fail(SVSB_E_INVALID, "svsb_launch_merge: NULL pointer");
    int rc;
    if ((int64_t)n_lists * stride > K_FAST_MAX && (rc = ws->ensure_merge_scratch((int64_t)n_lists * stride)) != SVSB_OK) return rc;
    CU(cudaSetDevice(ws->dev));
    CU(launch_merge((cudaStream_t)stream, (const u64*)d_keys, d_ids, d_counts, n_lists, stride, k,
                    ws->mscr_keys, ws->mscr_ids, d_out_scores, d_out_ids, d_out_count));
    return SVSB_OK;
}

extern "C" const char* svsb_last_error(void) { return g_err.c_str(); }
extern "C" const char* svsb_version(void) { return "svs_b200 0.1.0 (sm_100a)"; }
extern "C" int64_t svsb_launch_count(void) { return g_launches.load(); }
