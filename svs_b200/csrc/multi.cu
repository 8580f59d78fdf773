// Several devices in ONE process: what `svs_b200.install(svs, devices=[0, 1, ...])` / svsb_create(n_dev > 1) runs
// behind KB.retrieve (reference src/svs/kb.py:1608-1640 on a row-sharded matrix, SURVEY.md section 8e).
//
// Design.  The matrix is row-sharded in scan order (engine.cu: alloc_generation).  Every device gets a SHARD ENGINE --
// the very object a torchrun rank owns in the one-process-per-GPU deployment (gather window, stream, workspace) --
// and one host WORKER THREAD that does all the enqueueing for that device, so the host-side launch work of a query
// runs in parallel over the devices exactly as it does with one process per GPU.  A query is
//     every device:  [query staged from pinned host memory by a kernel] -> similarity -> selection whose epilogue
//                    pushes the k-candidate record into DEVICE 0's gather window (plain peer stores over NVLink /
//                    NVSwitch, published with a system-scope release store of the query's sequence number);
//     device 0:      merge kernel that acquires the `n_dev` flags of the window slot and writes the global top-k
//                    straight into pinned host memory.
// No copy-engine operation, no event hand-over between devices, no collective: the same fused exchange as
// svsb_query_peer (select.cu: peer_publish / merge_window_kernel), with device 0 as the only consumer.
// Up to TICKETS queries are in flight (svsb_query_submit / svsb_query_wait, or several caller threads): the window has
// 4 slots and a slot is reused only by query j + 4, whose submission required a ticket of query <= j + 1 to have been
// observed complete, i.e. merge(j) to have finished (device 0's stream runs the merges in sequence order).
// k > 2048 (the notebooks' n = len(kb) full ranking) and batches gather the per-device lists with peer copies instead
// and merge them on device 0 (merge_sorted_big_kernel / merge_lists_kernel); they run with the ticket queue drained.
#include "engine.cuh"

#include <chrono>
#include <functional>
#include <thread>

using namespace svsb;

namespace {

// One persistent thread per device.  run_all(job) runs job(i) on worker i for all i and returns the first failure.
// Workers spin for a short while after a job (a query loop posts the next job within a query time) before they sleep.
class WorkerPool {
public:
    WorkerPool(const std::vector<int>& devs) : devs_(devs), rc_(devs.size(), 0), err_(devs.size()) {
        for (size_t i = 0; i < devs.size(); ++i) th_.emplace_back([this, i] { loop((int)i); });
    }
    ~WorkerPool() {
        { std::lock_guard<std::mutex> lk(mu_); stop_ = true; epoch_.fetch_add(1, std::memory_order_release); }
        cv_go_.notify_all();
        for (auto& t : th_) t.join();
    }
    int run_all(const std::function<int(int)>& job) {
        job_ = &job;
        remaining_.store((int)th_.size(), std::memory_order_release);
        { std::lock_guard<std::mutex> lk(mu_); epoch_.fetch_add(1, std::memory_order_release); }
        cv_go_.notify_all();
        const auto t0 = std::chrono::steady_clock::now();
        int spins = 0;
        while (remaining_.load(std::memory_order_acquire) != 0) {
            if ((++spins & 63) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(200)) {
                std::unique_lock<std::mutex> lk(mu_);
                cv_done_.wait(lk, [this] { return remaining_.load(std::memory_order_acquire) == 0; });
                break;
            }
        }
        for (size_t i = 0; i < rc_.size(); ++i)
            if (rc_[i] != SVSB_OK) { g_err = err_[i]; return rc_[i]; }
        return SVSB_OK;
    }

private:
    void loop(int idx) {
        cudaSetDevice(devs_[idx]);
        unsigned long long seen = 0;
        while (true) {
            const auto t0 = std::chrono::steady_clock::now();
            int spins = 0;
            while (epoch_.load(std::memory_order_acquire) == seen) {
                if ((++spins & 63) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(300)) {
                    std::unique_lock<std::mutex> lk(mu_);
                    cv_go_.wait(lk, [&] { return epoch_.load(std::memory_order_acquire) != seen; });
                    break;
                }
            }
            seen = epoch_.load(std::memory_order_acquire);
            if (stop_) return;
            const int r = (*job_)(idx);
            rc_[idx] = r;
            if (r != SVSB_OK) err_[idx] = g_err;
            if (remaining_.fetch_sub(1, std::memory_order_acq_rel) == 1) {
                std::lock_guard<std::mutex> lk(mu_);
                cv_done_.notify_all();
            }
        }
    }
    std::vector<int> devs_;
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_go_, cv_done_;
    std::atomic<unsigned long long> epoch_{0};
    std::atomic<int> remaining_{0};
    const std::function<int(int)>* job_ = nullptr;
    std::vector<int> rc_;
    std::vector<std::string> err_;
    bool stop_ = false;
};

constexpr int TICKETS = 3;

}  // namespace

struct svsb_ticket {
    float* h_q = nullptr; int q_cap = 0;           // pinned + portable: every device's staging kernel reads it over PCIe
    float* h_scores = nullptr; int64_t* h_ids = nullptr; int32_t* h_count = nullptr;    // pinned: device 0's merge writes them
    float* d_scores = nullptr; int64_t* d_ids = nullptr; int32_t* d_count = nullptr;    // device 0: bench (device-resident) outputs
    cudaEvent_t ev = nullptr;                      // device 0's stream: this ticket's merge is done
    bool busy = false;
    int64_t kk = 0;
    std::shared_ptr<Generation> gen;               // the generation the query runs on stays alive until the ticket is released
};

struct KidScratch {                                // per device: operands of the batched and the large-k path
    float* dQ = nullptr; int64_t dQ_cap = 0;
    int64_t* rec = nullptr; int64_t rec_cap = 0;
    cudaEvent_t ev = nullptr;
};

struct Multi {
    std::vector<svsb_engine*> kids;
    std::vector<KidScratch> scratch;
    std::unique_ptr<WorkerPool> pool;
    std::mutex mu;                                 // one submission at a time: all devices see the same sequence
    std::condition_variable cv;
    unsigned long long seq = 0;
    svsb_ticket tk[TICKETS];
    // device 0: gathered lists + outputs of the large-k / batched paths, pinned staging for their results
    u64* g_keys = nullptr; int64_t* g_ids = nullptr; int64_t g_cap = 0; int32_t* g_counts = nullptr;
    float* m_scores = nullptr; int64_t* m_ids = nullptr; int32_t* m_count = nullptr; int64_t m_cap = 0;
    int64_t* g_rec = nullptr; int64_t g_rec_cap = 0;
    float* b_scores = nullptr; int64_t* b_ids = nullptr; int32_t* b_counts = nullptr; int64_t b_cap = 0, b_cnt_cap = 0;
    float* h_big_scores = nullptr; int64_t* h_big_ids = nullptr; int64_t h_big_cap = 0; int32_t* h_big_count = nullptr;
    float* h_Q = nullptr; int64_t h_Q_cap = 0;     // pinned staging of a batch's queries (read by every device)
    u64* b_sk = nullptr; int64_t* b_sp = nullptr; int64_t b_scr_cap = 0;   // the batch merge's own scratch (fused merges in flight use device 0's)
    std::vector<cudaEvent_t> kev;                  // bench: similarity-kernel brackets on device 0
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    svsb_ticket* last = nullptr;                   // bench: ticket holding the last result
};

static inline int root_dev(const Multi* m) { return m->kids[0]->devs[0]; }

int multi_create(svsb_engine* e) {
    const int nd = (int)e->devs.size();
    std::unique_ptr<Multi> m(new Multi());
    e->multi = m.get();                            // owned by the engine from here on (multi_destroy releases what exists)
    m.release();
    Multi* M = e->multi;
    M->scratch.resize(nd);
    for (int i = 0; i < nd; ++i) {
        svsb_engine* kid = nullptr;
        int dev = e->devs[i];
        int rc = engine_create(&dev, 1, /*as_kid=*/true, &kid);
        if (rc != SVSB_OK) return rc;
        M->kids.push_back(kid);
        if ((rc = svsb_xchg_create(kid, nd, i, K_FAST_MAX, nullptr)) != SVSB_OK) return rc;
        CU(cudaSetDevice(dev));
        CU(cudaEventCreateWithFlags(&M->scratch[i].ev, cudaEventDisableTiming));
    }
    for (int i = 0; i < nd; ++i) {
        int rc = svsb_xchg_connect_local(M->kids[i], M->kids.data());
        if (rc != SVSB_OK) return rc;
    }
    CU(cudaSetDevice(root_dev(M)));
    for (auto& t : M->tk) {
        CU(cudaHostAlloc(&t.h_scores, (size_t)K_FAST_MAX * 4, cudaHostAllocPortable));
        CU(cudaHostAlloc(&t.h_ids, (size_t)K_FAST_MAX * 8, cudaHostAllocPortable));
        CU(cudaHostAlloc(&t.h_count, 64, cudaHostAllocPortable));
        CU(cudaMalloc(&t.d_scores, (size_t)K_FAST_MAX * 4));
        CU(cudaMalloc(&t.d_ids, (size_t)K_FAST_MAX * 8));
        CU(cudaMalloc(&t.d_count, 64));
        CU(cudaEventCreateWithFlags(&t.ev, cudaEventDisableTiming));
    }
    CU(cudaMalloc(&M->g_counts, (size_t)nd * 4));
    CU(cudaMalloc(&M->m_count, 64));
    CU(cudaHostAlloc(&M->h_big_count, 64, cudaHostAllocPortable));
    CU(cudaEventCreate(&M->ev0));
    CU(cudaEventCreate(&M->ev1));
    M->pool.reset(new WorkerPool(e->devs));
    return SVSB_OK;
}

void multi_destroy(svsb_engine* e) {
    Multi* m = e->multi;
    if (!m) return;
    m->pool.reset();                               // joins the workers
    for (size_t i = 0; i < m->kids.size(); ++i) {
        if (!m->kids[i]) continue;
        cudaSetDevice(m->kids[i]->devs[0]);
        cudaDeviceSynchronize();
        KidScratch& ks = m->scratch[i];
        if (ks.dQ) cudaFree(ks.dQ);
        if (ks.rec) cudaFree(ks.rec);
        if (ks.ev) cudaEventDestroy(ks.ev);
    }
    if (!m->kids.empty()) {
        cudaSetDevice(root_dev(m));
        for (auto& t : m->tk) {
            if (t.h_q) cudaFreeHost(t.h_q);
            if (t.h_scores) cudaFreeHost(t.h_scores);
            if (t.h_ids) cudaFreeHost(t.h_ids);
            if (t.h_count) cudaFreeHost(t.h_count);
            if (t.d_scores) cudaFree(t.d_scores);
            if (t.d_ids) cudaFree(t.d_ids);
            if (t.d_count) cudaFree(t.d_count);
            if (t.ev) cudaEventDestroy(t.ev);
        }
        void* dp[] = {m->g_keys, m->g_ids, m->g_counts, m->m_scores, m->m_ids, m->m_count, m->g_rec, m->b_scores, m->b_ids, m->b_counts,
                      m->b_sk, m->b_sp};
        for (void* p : dp) if (p) cudaFree(p);
        void* hp[] = {m->h_big_scores, m->h_big_ids, m->h_big_count, m->h_Q};
        for (void* p : hp) if (p) cudaFreeHost(p);
        for (auto ev : m->kev) cudaEventDestroy(ev);
        if (m->ev0) cudaEventDestroy(m->ev0);
        if (m->ev1) cudaEventDestroy(m->ev1);
    }
    // every device stops pushing before any window is freed
    for (auto* kid : m->kids) if (kid) svsb_xchg_disconnect(kid);
    for (auto* kid : m->kids) if (kid) svsb_destroy(kid);
    delete m;
    e->multi = nullptr;
}

// Per-device views of generation g + every buffer the fused path uses, sized NOW: allocations are implicit
// synchronisation points and must not land between the enqueueing of one query on two devices (a merge kernel
// spinning for a peer whose kernels wait behind a cudaMalloc never ends -- DESIGN.md section 4, K6).
int multi_publish(svsb_engine* e, const std::shared_ptr<Generation>& g) {
    Multi* m = e->multi;
    const int nd = (int)m->kids.size();
    // m->mu: no query is half-enqueued while the buffers below are (re)allocated.  Queries already in flight are fully
    // enqueued and keep running; a cudaFree of a buffer they use waits for them.  (Not a wait for the tickets themselves:
    // a caller may hold a pending svsb_query_submit handle while it loads.)
    std::unique_lock<std::mutex> lk(m->mu);
    g->child_gen.clear();
    for (int i = 0; i < nd; ++i) {
        std::shared_ptr<Generation> cg(new Generation());
        const Shard& s = g->shards[i];
        cg->id = g->id; cg->n = s.n; cg->n_live = s.n_live; cg->d = g->d; cg->ld = g->ld; cg->norm_mode = g->norm_mode;
        cg->owns_live = false;                     // the parent generation owns the tombstone arrays
        cg->max_dev = g->max_dev; cg->n_out_of_tol = g->n_out_of_tol;
        cg->shards.push_back(s);
        g->child_gen.push_back(cg);
    }
    return m->pool->run_all([&](int i) -> int {
        svsb_engine* kid = m->kids[i];
        Xchg* x = kid->xchg.get();
        const Shard& s = g->shards[i];
        CU(cudaSetDevice(s.dev));
        int rc;
        if (s.n > 0 && (rc = x->ws.ensure_rows(s.n)) != SVSB_OK) return rc;
        if (g->ld > 0 && (rc = x->ws.ensure_q(g->ld)) != SVSB_OK) return rc;
        if ((rc = x->ws.ensure_out(K_FAST_MAX)) != SVSB_OK) return rc;
        if (i == 0 && (rc = x->ws.ensure_merge_scratch((int64_t)nd * K_FAST_MAX)) != SVSB_OK) return rc;
        // the fused path is software-pipelined per device: two workspace sets alternate, selection + push run on a side stream
        if (!kid->side_st) CU(cudaStreamCreateWithFlags(&kid->side_st, cudaStreamNonBlocking));
        if (kid->shard_ws.size() < 2) kid->shard_ws.resize(2);
        if (kid->sel_pending.size() < 2) kid->sel_pending.resize(2, 0);
        for (int t = 0; t < 2; ++t) {
            if (!kid->shard_ws[t]) { kid->shard_ws[t].reset(new DevWs()); kid->shard_ws[t]->dev = s.dev; }
            DevWs& w = *kid->shard_ws[t];
            if (s.n > 0 && (rc = w.ensure_rows(s.n)) != SVSB_OK) return rc;
            if (g->ld > 0 && (rc = w.ensure_q(g->ld)) != SVSB_OK) return rc;
            if ((rc = w.ensure_out(K_FAST_MAX)) != SVSB_OK) return rc;
            if (!w.ev) CU(cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming));
            if (!w.ev_sel) CU(cudaEventCreateWithFlags(&w.ev_sel, cudaEventDisableTiming));
        }
        return SVSB_OK;
    });
}

// ------------------------------------------------------------------------------------------------
// the fused path: k <= 2048, one query
// ------------------------------------------------------------------------------------------------
struct FastJob {
    const Generation* g = nullptr;
    unsigned long long seq = 0;
    int64_t kk = 0;
    const float* h_q = nullptr;                    // pinned host query, staged on every device by a kernel ...
    float* const* d_q = nullptr; int64_t q_off = 0; // ... or device-resident queries (bench): d_q[i] + q_off on device i
    float* out_scores = nullptr; int64_t* out_ids = nullptr; int32_t* out_count = nullptr;
    cudaEvent_t ev_done = nullptr;
    cudaEvent_t kev0 = nullptr, kev1 = nullptr;    // optional bracket of device 0's similarity kernel
};

// Per device, software-pipelined like the one-process-per-GPU loop (engine.cu: svsb_enqueue_query_peer): the similarity
// pass of query j runs on the device's main stream with one SM left free, its selection + push on the side stream on
// that SM, so query j+1's matrix pass overlaps query j's selection, push and (device 0) merge.  Two workspace sets
// alternate; ev_sel of a set gates the similarity pass two queries on.
static int kid_fast(Multi* m, int i, const FastJob& j) {
    svsb_engine* kid = m->kids[i];
    Xchg* x = kid->xchg.get();
    Xchg* xr = m->kids[0]->xchg.get();
    const Generation* cg = j.g->child_gen[i].get();
    const Shard& s = cg->shards[0];
    const int set = (int)(j.seq & 1);
    DevWs& w = *kid->shard_ws[set];
    cudaStream_t st = x->st, side = kid->side_st;
    CU(cudaSetDevice(s.dev));
    const int slot = (int)(j.seq % (unsigned long long)xr->slots);
    PeerPush push{};
    push.world = 1; push.cap = xr->cap; push.seq = j.seq;        // one consumer: device 0's window
    push.rec[0] = xr->rec_of(xr->block, slot, i);
    push.flag[0] = xr->flags_of(xr->block, slot) + i;
    if (s.n_live == 0) {
        CU(launch_push_empty(side, push));
        return SVSB_OK;
    }
    const int shift = group_shift_for(s.n);
    const bool pipelined = sm_count(s.dev) > 8;
    if (kid->sel_pending[set]) CU(cudaStreamWaitEvent(st, w.ev_sel, 0));   // the set's previous selection is done with it
    const float* dq = j.d_q ? j.d_q[i] + j.q_off : w.d_q;
    if (!j.d_q) CU(launch_stage_query(st, j.h_q, w.d_q, cg->ld));
    if (i == 0 && j.kev0) CU(cudaEventRecord(j.kev0, st));
    w.gmax_dirty = true;
    {   // the similarity kernel streams its first tiles under the staging kernel (programmatic dependent launch)
        PdlScope pdl(!j.d_q && env_int("SVSB_PDL", 1) != 0);
        CU(launch_gemv(st, s.dev, s.M, s.n, cg->d, cg->ld, dq, w.scores, w.gmax, shift, 0, 0, 0, pipelined ? 1 : 0, s.live));
    }
    if (i == 0 && j.kev1) CU(cudaEventRecord(j.kev1, st));
    CU(cudaEventRecord(w.ev, st));
    CU(cudaStreamWaitEvent(side, w.ev, 0));
    CU(launch_select(side, w.scores, s.n, w.gmax, shift, (int)std::min<int64_t>(j.kk, s.n_live), s.ids, s.row0, w.cand, w.cand_cap,
                     w.out_keys, w.out_scores, w.out_ids, w.out_count, nullptr, &push));
    w.gmax_dirty = false;
    CU(cudaEventRecord(w.ev_sel, side));
    kid->sel_pending[set] = 1;
    return SVSB_OK;
}

// Device 0's waiting merge, enqueued (on device 0's side stream) by the submitting thread AFTER every device's
// selection with its push has been enqueued: a kernel that waits is only ever launched behind everything it waits for,
// so no host-side operation with an implicit device synchronisation (cudaMalloc / cudaFree of a concurrent load, ...)
// can come between a spinning merge and the launch of a push it needs -- with several virtual shards on ONE device that
// would otherwise deadlock until the merge's timeout.
static int root_merge(Multi* m, const FastJob& j) {
    svsb_engine* root = m->kids[0];
    Xchg* xr = root->xchg.get();
    DevWs& w = xr->ws;
    cudaStream_t st = root->side_st;
    const int nd = (int)m->kids.size();
    const int slot = (int)(j.seq % (unsigned long long)xr->slots);
    CU(cudaSetDevice(root_dev(m)));
    u64* sk = nullptr; int64_t* sp = nullptr;
    if ((int64_t)nd * j.kk > K_FAST_MAX) { sk = w.mscr_keys; sp = w.mscr_ids; }
    CU(launch_merge_window(st, xr->rec_of(xr->block, slot, 0), xr->flags_of(xr->block, slot), j.seq, nd, xr->cap, (int)j.kk,
                           xr->timeout_ns, sk, sp, j.out_scores, j.out_ids, j.out_count));
    CU(cudaEventRecord(j.ev_done, st));
    return SVSB_OK;
}

// caller holds m->mu: a ticket nobody uses (blocks until one is released)
static svsb_ticket* free_ticket_locked(Multi* m, std::unique_lock<std::mutex>& lk) {
    svsb_ticket* t = nullptr;
    // other threads release tickets within a query time; a caller that already holds every ticket as a pending handle
    // would wait for itself -- give up with an error instead
    const bool ok = m->cv.wait_for(lk, std::chrono::milliseconds(env_int("SVSB_SUBMIT_TIMEOUT_MS", 5000)),
                                   [&] { for (auto& c : m->tk) if (!c.busy) { t = &c; return true; } return false; });
    return ok ? t : nullptr;
}

// caller holds m->mu and got `t` from free_ticket_locked without releasing the lock since
static int submit_locked(Multi* m, svsb_ticket* t, FastJob& j, bool host_out) {
    t->busy = true; t->kk = j.kk;
    if (host_out) { *t->h_count = -1; j.out_scores = t->h_scores; j.out_ids = t->h_ids; j.out_count = t->h_count; }
    else { j.out_scores = t->d_scores; j.out_ids = t->d_ids; j.out_count = t->d_count; }
    j.ev_done = t->ev;
    j.seq = ++m->seq;
    int rc = m->pool->run_all([&](int i) { return kid_fast(m, i, j); });
    if (rc == SVSB_OK) rc = root_merge(m, j);
    if (rc != SVSB_OK) { t->busy = false; t->gen.reset(); m->cv.notify_all(); }
    return rc;
}

static int ticket_wait(Multi* m, svsb_ticket* t) {
    CU(cudaSetDevice(root_dev(m)));
    CU(cudaEventSynchronize(t->ev));
    return SVSB_OK;
}
static void ticket_release(Multi* m, svsb_ticket* t) {
    { std::lock_guard<std::mutex> lk(m->mu); t->busy = false; t->gen.reset(); }
    m->cv.notify_all();
}

static int multi_query_big(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int64_t kk,
                           float* out_scores, int64_t* out_ids, int32_t* out_count);

int multi_submit(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int64_t kk, svsb_ticket** out) {
    Multi* m = e->multi;
    std::unique_lock<std::mutex> lk(m->mu);
    svsb_ticket* t = free_ticket_locked(m, lk);
    if (!t) return fail(SVSB_E_STATE, "svsb_query_submit: 3 queries are pending already (wait for the oldest first)");
    if (g->ld > t->q_cap) {                        // this ticket is free and nothing is half-enqueued (we hold m->mu)
        CU(cudaSetDevice(root_dev(m)));
        if (t->h_q) cudaFreeHost(t->h_q);
        t->h_q = nullptr; t->q_cap = 0;
        CU(cudaHostAlloc(&t->h_q, (size_t)g->ld * 4, cudaHostAllocPortable));
        t->q_cap = g->ld;
    }
    memcpy(t->h_q, q, (size_t)d * 4);
    for (int i = d; i < g->ld; ++i) t->h_q[i] = 0.f;
    t->gen = g;
    FastJob j; j.g = g.get(); j.kk = kk; j.h_q = t->h_q;
    const int rc = submit_locked(m, t, j, /*host_out=*/true);
    if (rc == SVSB_OK) *out = t;
    return rc;
}

int multi_wait(svsb_engine* e, svsb_ticket* t, float* out_scores, int64_t* out_ids, int32_t* out_count) {
    Multi* m = e->multi;
    int rc = ticket_wait(m, t);
    if (rc == SVSB_OK) {
        const int32_t cnt = *t->h_count;
        if (cnt == MERGE_WINDOW_TIMED_OUT) rc = fail(SVSB_E_STATE, "a device's candidate record did not arrive in time");
        else if (cnt < 0 || cnt > t->kk) rc = fail(SVSB_E_CUDA, "internal: merge returned a bad count");
        else {
            memcpy(out_scores, t->h_scores, (size_t)cnt * 4);
            memcpy(out_ids, t->h_ids, (size_t)cnt * 8);
            *out_count = cnt;
        }
    }
    ticket_release(m, t);
    return rc;
}

int multi_query(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int64_t kk,
                float* out_scores, int64_t* out_ids, int32_t* out_count) {
    if (kk > K_FAST_MAX) return multi_query_big(e, g, q, d, kk, out_scores, out_ids, out_count);
    svsb_ticket* t = nullptr;
    int rc = multi_submit(e, g, q, d, kk, &t);
    if (rc != SVSB_OK) return rc;
    return multi_wait(e, t, out_scores, out_ids, out_count);
}

// ------------------------------------------------------------------------------------------------
// k > 2048: per-device sorted lists (full sort of the shard's keys), gathered with peer copies, rank-merged on device 0
// ------------------------------------------------------------------------------------------------
static int copy_to_root(Multi* m, int i, void* dst, const void* src, size_t bytes, cudaStream_t root_st) {
    const int rd = root_dev(m), kd = m->kids[i]->devs[0];
    if (bytes == 0) return SVSB_OK;
    if (kd == rd) CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, root_st));
    else CU(cudaMemcpyPeerAsync(dst, rd, src, kd, bytes, root_st));
    return SVSB_OK;
}

static int multi_query_big(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* q, int32_t d, int64_t kk,
                           float* out_scores, int64_t* out_ids, int32_t* out_count) {
    Multi* m = e->multi;
    const int nd = (int)m->kids.size();
    std::unique_lock<std::mutex> lk(m->mu);        // exclusive use of the gather scratch; fused queries in flight keep running
    CU(cudaSetDevice(root_dev(m)));
    if (g->ld > m->h_Q_cap) {
        if (m->h_Q) cudaFreeHost(m->h_Q);
        m->h_Q = nullptr; m->h_Q_cap = 0;
        CU(cudaHostAlloc(&m->h_Q, (size_t)g->ld * 4, cudaHostAllocPortable));
        m->h_Q_cap = g->ld;
    }
    float* hq = m->h_Q;
    memcpy(hq, q, (size_t)d * 4);
    for (int i = d; i < g->ld; ++i) hq[i] = 0.f;
    if (kk > m->g_cap) {
        void* ptrs[] = {m->g_keys, m->g_ids, m->m_scores, m->m_ids};
        for (void* p : ptrs) if (p) cudaFree(p);
        m->g_keys = nullptr; m->g_ids = nullptr; m->m_scores = nullptr; m->m_ids = nullptr; m->g_cap = 0;
        CU(cudaMalloc(&m->g_keys, (size_t)nd * kk * 8));
        CU(cudaMalloc(&m->g_ids, (size_t)nd * kk * 8));
        CU(cudaMalloc(&m->m_scores, (size_t)kk * 4));
        CU(cudaMalloc(&m->m_ids, (size_t)kk * 8));
        m->g_cap = kk;
    }
    if (kk > m->h_big_cap) {
        if (m->h_big_scores) cudaFreeHost(m->h_big_scores);
        if (m->h_big_ids) cudaFreeHost(m->h_big_ids);
        m->h_big_scores = nullptr; m->h_big_ids = nullptr; m->h_big_cap = 0;
        CU(cudaHostAlloc(&m->h_big_scores, (size_t)kk * 4, cudaHostAllocPortable));
        CU(cudaHostAlloc(&m->h_big_ids, (size_t)kk * 8, cudaHostAllocPortable));
        m->h_big_cap = kk;
    }
    int rc = m->pool->run_all([&](int i) -> int {
        svsb_engine* kid = m->kids[i];
        Xchg* x = kid->xchg.get();
        const Generation* cg = g->child_gen[i].get();
        const Shard& s = cg->shards[0];
        DevWs& w = x->ws;
        CU(cudaSetDevice(s.dev));
        if (s.n_live > 0) {
            const int64_t kl = std::min(kk, s.n_live);
            int rc2 = prepare_ws(w, cg, s, kl);
            if (rc2 != SVSB_OK) return rc2;
            const int shift = group_shift_for(s.n);
            CU(cudaMemcpyAsync(w.d_q, hq, (size_t)cg->ld * 4, cudaMemcpyHostToDevice, x->st));
            w.gmax_dirty = true;
            CU(launch_gemv(x->st, s.dev, s.M, s.n, cg->d, cg->ld, w.d_q, w.scores, w.gmax, shift, 0, 0, 0, 0, s.live));
            if (kl <= K_FAST_MAX)
                CU(launch_select(x->st, w.scores, s.n, w.gmax, shift, (int)kl, s.ids, s.row0, w.cand, w.cand_cap,
                                 w.out_keys, w.out_scores, w.out_ids, w.out_count));
            else
                CU(launch_fullsort_topk(x->st, w.scores, s.n, w.gmax, shift, kl, s.ids, s.row0, w.sortbuf,
                                        w.out_keys, w.out_scores, w.out_ids, w.out_count));
            w.gmax_dirty = false;
        }
        CU(cudaEventRecord(m->scratch[i].ev, x->st));
        return SVSB_OK;
    });
    if (rc != SVSB_OK) return rc;
    CU(cudaSetDevice(root_dev(m)));
    cudaStream_t rst = m->kids[0]->xchg->st;
    for (int i = 0; i < nd; ++i) {
        const Shard& s = g->shards[i];
        DevWs& w = m->kids[i]->xchg->ws;
        if (i != 0) CU(cudaStreamWaitEvent(rst, m->scratch[i].ev, 0));
        if (s.n_live == 0) { CU(cudaMemsetAsync(m->g_counts + i, 0, 4, rst)); continue; }
        const int64_t kl = std::min(kk, s.n_live);
        if ((rc = copy_to_root(m, i, m->g_keys + (int64_t)i * kk, w.out_keys, (size_t)kl * 8, rst)) != SVSB_OK) return rc;
        if ((rc = copy_to_root(m, i, m->g_ids + (int64_t)i * kk, w.out_ids, (size_t)kl * 8, rst)) != SVSB_OK) return rc;
        if ((rc = copy_to_root(m, i, m->g_counts + i, w.out_count, 4, rst)) != SVSB_OK) return rc;
    }
    CU(launch_merge_sorted_big(rst, m->g_keys, m->g_ids, m->g_counts, nd, kk, kk, 1, kk, m->m_scores, m->m_ids, m->m_count));
    CU(cudaMemcpyAsync(m->h_big_scores, m->m_scores, (size_t)kk * 4, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpyAsync(m->h_big_ids, m->m_ids, (size_t)kk * 8, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpyAsync(m->h_big_count, m->m_count, 4, cudaMemcpyDeviceToHost, rst));
    CU(cudaStreamSynchronize(rst));
    // the copies above read the other devices' buffers: those devices may go on only now
    const int32_t cnt = *m->h_big_count;
    if (cnt != (int32_t)kk) return fail(SVSB_E_CUDA, "internal: large-k merge returned a bad count");
    memcpy(out_scores, m->h_big_scores, (size_t)cnt * 4);
    memcpy(out_ids, m->h_big_ids, (size_t)cnt * 8);
    *out_count = cnt;
    return SVSB_OK;
}

// ------------------------------------------------------------------------------------------------
// batches: every device runs the batched pipeline on its shard (tensor-core coarse pass + exact refine, or the exact
// multi-query / single-query kernels -- engine.cu: batch_local_records_gen), the b records per device are gathered
// on device 0 with one peer copy each and merged by ONE launch (a CTA per query)
// ------------------------------------------------------------------------------------------------
int multi_query_batch(svsb_engine* e, const std::shared_ptr<Generation>& g, const float* Q, int32_t b, int32_t d, int32_t k,
                      float* out_scores, int64_t* out_ids, int32_t* out_counts) {
    Multi* m = e->multi;
    const int nd = (int)m->kids.size();
    const int64_t kk = std::min<int64_t>(k, g->n_live);
    if (kk > K_FAST_MAX) {                          // full rankings: one large-k query at a time
        for (int32_t i = 0; i < b; ++i) {
            int rc = multi_query_big(e, g, Q + (int64_t)i * d, d, kk, out_scores + (int64_t)i * k, out_ids + (int64_t)i * k, out_counts + i);
            if (rc != SVSB_OK) return rc;
        }
        return SVSB_OK;
    }
    std::unique_lock<std::mutex> lk(m->mu);        // exclusive use of the gather scratch; fused queries in flight keep running
    const int kr = (int)kk;                         // entries per record
    const int64_t rec = RecordView{nullptr, kr}.words();
    const int ld = g->ld;
    CU(cudaSetDevice(root_dev(m)));
    if ((int64_t)b * ld > m->h_Q_cap) {
        if (m->h_Q) cudaFreeHost(m->h_Q);
        m->h_Q = nullptr; m->h_Q_cap = 0;
        CU(cudaHostAlloc(&m->h_Q, (size_t)b * ld * 4, cudaHostAllocPortable));
        m->h_Q_cap = (int64_t)b * ld;
    }
    stage_queries(m->h_Q, Q, b, d, ld);
    if ((int64_t)nd * b * rec > m->g_rec_cap) {
        if (m->g_rec) cudaFree(m->g_rec);
        m->g_rec = nullptr; m->g_rec_cap = 0;
        CU(cudaMalloc(&m->g_rec, (size_t)nd * b * rec * 8));
        m->g_rec_cap = (int64_t)nd * b * rec;
    }
    if ((int64_t)b * kr > m->b_cap || b > m->b_cnt_cap) {
        void* ptrs[] = {m->b_scores, m->b_ids, m->b_counts};
        for (void* p : ptrs) if (p) cudaFree(p);
        m->b_scores = nullptr; m->b_ids = nullptr; m->b_counts = nullptr; m->b_cap = 0; m->b_cnt_cap = 0;
        CU(cudaMalloc(&m->b_scores, (size_t)b * kr * 4));
        CU(cudaMalloc(&m->b_ids, (size_t)b * kr * 8));
        CU(cudaMalloc(&m->b_counts, (size_t)b * 4));
        m->b_cap = (int64_t)b * kr; m->b_cnt_cap = b;
    }
    int rc;
    if ((int64_t)nd * kr > K_FAST_MAX && (int64_t)b * nd * kr > m->b_scr_cap) {
        if (m->b_sk) cudaFree(m->b_sk);
        if (m->b_sp) cudaFree(m->b_sp);
        m->b_sk = nullptr; m->b_sp = nullptr; m->b_scr_cap = 0;
        CU(cudaMalloc(&m->b_sk, (size_t)b * nd * kr * 8));
        CU(cudaMalloc(&m->b_sp, (size_t)b * nd * kr * 8));
        m->b_scr_cap = (int64_t)b * nd * kr;
    }
    rc = m->pool->run_all([&](int i) -> int {
        svsb_engine* kid = m->kids[i];
        KidScratch& ks = m->scratch[i];
        cudaStream_t st = kid->xchg->st;
        CU(cudaSetDevice(kid->devs[0]));
        if ((int64_t)b * ld > ks.dQ_cap) {
            if (ks.dQ) cudaFree(ks.dQ);
            ks.dQ = nullptr; ks.dQ_cap = 0;
            CU(cudaMalloc(&ks.dQ, (size_t)b * ld * 4));
            ks.dQ_cap = (int64_t)b * ld;
        }
        if ((int64_t)b * rec > ks.rec_cap) {
            if (ks.rec) cudaFree(ks.rec);
            ks.rec = nullptr; ks.rec_cap = 0;
            CU(cudaMalloc(&ks.rec, (size_t)b * rec * 8));
            ks.rec_cap = (int64_t)b * rec;
        }
        CU(cudaMemcpyAsync(ks.dQ, m->h_Q, (size_t)b * ld * 4, cudaMemcpyHostToDevice, st));
        int32_t nfb = 0;
        int rc2 = batch_local_records_gen(kid, g->child_gen[i], st, ks.dQ, b, kr, ks.rec, &nfb);
        if (rc2 != SVSB_OK) return rc2;
        CU(cudaEventRecord(ks.ev, st));
        return SVSB_OK;
    });
    if (rc != SVSB_OK) return rc;
    CU(cudaSetDevice(root_dev(m)));
    cudaStream_t rst = m->kids[0]->xchg->st;
    for (int i = 0; i < nd; ++i) {
        if (i != 0) CU(cudaStreamWaitEvent(rst, m->scratch[i].ev, 0));
        if ((rc = copy_to_root(m, i, m->g_rec + (int64_t)i * b * rec, m->scratch[i].rec, (size_t)b * rec * 8, rst)) != SVSB_OK) return rc;
    }
    u64* sk = nullptr; int64_t* sp = nullptr;
    if ((int64_t)nd * kr > K_FAST_MAX) { sk = m->b_sk; sp = m->b_sp; }
    if ((rc = merge_records(rst, RecordView{m->g_rec, kr}, nd, (int64_t)b * rec, b, kr, sk, sp, m->b_scores, m->b_ids, m->b_counts)) != SVSB_OK)
        return rc;
    // results: (b, kr) on the device, (b, k) at the caller
    CU(cudaMemcpy2DAsync(out_scores, (size_t)k * 4, m->b_scores, (size_t)kr * 4, (size_t)kr * 4, (size_t)b, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpy2DAsync(out_ids, (size_t)k * 8, m->b_ids, (size_t)kr * 8, (size_t)kr * 8, (size_t)b, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpyAsync(out_counts, m->b_counts, (size_t)b * 4, cudaMemcpyDeviceToHost, rst));
    CU(cudaStreamSynchronize(rst));
    return SVSB_OK;
}

// ------------------------------------------------------------------------------------------------
// pairwise top pairs: every device runs its share of the static plan (engine.cu: pairs_plan) -- the triangle of its own
// shard and rectangles against 1024-row blocks of its peers' fp16 rows, copied over -- with its OWN running threshold.
// That is valid: the n-th largest coarse score over a subset of the pairs is at most the n-th largest over all pairs,
// so no pair of the exact top n is dropped.  Each device re-scores its survivors exactly (the second row read over the
// peer mapping; the bits do not depend on the device) and keeps its top min(n, survivors) in the final order; device 0
// gathers the lists and rank-merges them.  No kernel waits on a flag: devices are ordered by events and stream waits.
// ------------------------------------------------------------------------------------------------
int multi_top_pairs(svsb_engine* e, const std::shared_ptr<Generation>& g, int64_t n, float eps2, float* out_scores,
                    int64_t* out_ids_a, int64_t* out_ids_b, int64_t* out_count) {
    Multi* m = e->multi;
    const int nd = (int)m->kids.size();
    std::unique_lock<std::mutex> lk(m->mu);        // exclusive use of the kids' batch workspaces; fused queries in flight keep running
    std::vector<Generation*> views;
    std::vector<int64_t> shard_rows;
    for (int i = 0; i < nd; ++i) { views.push_back(g->child_gen[i].get()); shard_rows.push_back(g->shards[i].n); }
    const PairRows rows = pair_rows_of(views);
    const std::vector<std::vector<PairTask>> plan = pairs_plan(shard_rows);
    std::vector<PairsDev> r((size_t)nd);
    // fixed-size buffers and every device's fp16 shadow first: the coarse pass copies blocks of its peers' shadows
    int rc = m->pool->run_all([&](int i) { return pairs_dev_prepare(m->kids[i], views[i], n, eps2, r[i]); });
    if (rc != SVSB_OK) return rc;
    std::vector<PairShadow> shadows;
    for (const Generation* v : views) shadows.push_back(PairShadow{v->M16, v->shards[0].dev});
    rc = m->pool->run_all([&](int i) { return pairs_dev_coarse(r[i], i, plan[i], shadows, rows); });   // ends with every device idle
    if (rc != SVSB_OK) return rc;
    // every buffer sized by the survivor counts, on every device, before the re-score reads peer rows
    int64_t stride = 0, total = 0;
    for (auto& x : r) { stride = std::max(stride, std::min(n, x.C)); total += std::min(n, x.C); }
    if (total < n) return fail(SVSB_E_CUDA, "internal: pair lists shorter than the requested count");
    rc = m->pool->run_all([&](int i) { return pairs_dev_alloc(r[i]); });
    if (rc != SVSB_OK) return rc;
    const int rd = root_dev(m);
    CU(cudaSetDevice(rd));
    DevBufs bufs; bufs.dev = rd;
    float* l_scores; int64_t* l_a; int64_t* l_b; int32_t* l_cnt; float* o_scores; int64_t* o_a; int64_t* o_b; int32_t* o_cnt;
    CU(bufs.get(&l_scores, (size_t)(nd * stride))); CU(bufs.get(&l_a, (size_t)(nd * stride))); CU(bufs.get(&l_b, (size_t)(nd * stride)));
    CU(bufs.get(&l_cnt, (size_t)nd));
    CU(bufs.get(&o_scores, (size_t)n)); CU(bufs.get(&o_a, (size_t)n)); CU(bufs.get(&o_b, (size_t)n)); CU(bufs.get(&o_cnt, 16));
    rc = m->pool->run_all([&](int i) -> int {
        if (r[i].kl == 0) return SVSB_OK;
        int rc2 = pairs_dev_finish(r[i], rows, nullptr);                      // global rows: device 0 maps them to ids
        if (rc2 != SVSB_OK) return rc2;
        CU(cudaEventRecord(m->scratch[i].ev, r[i].st));
        return SVSB_OK;
    });
    if (rc != SVSB_OK) return rc;
    CU(cudaSetDevice(rd));
    cudaStream_t rst = m->kids[0]->xchg->st;
    for (int i = 0; i < nd; ++i) {
        const int64_t kl = r[i].kl;
        if (kl == 0) { CU(cudaMemsetAsync(l_cnt + i, 0, 4, rst)); continue; }
        CU(cudaStreamWaitEvent(rst, m->scratch[i].ev, 0));
        if ((rc = copy_to_root(m, i, l_scores + i * stride, r[i].o_scores, (size_t)kl * 4, rst)) != SVSB_OK) return rc;
        if ((rc = copy_to_root(m, i, l_a + i * stride, r[i].o_a, (size_t)kl * 8, rst)) != SVSB_OK) return rc;
        if ((rc = copy_to_root(m, i, l_b + i * stride, r[i].o_b, (size_t)kl * 8, rst)) != SVSB_OK) return rc;
        if ((rc = copy_to_root(m, i, l_cnt + i, r[i].o_cnt, 4, rst)) != SVSB_OK) return rc;
    }
    CU(launch_merge_sorted_pairs(rst, l_scores, l_a, l_b, l_cnt, nd, stride, n, rows, o_scores, o_a, o_b, o_cnt));
    int32_t cnt = 0;
    CU(cudaMemcpyAsync(out_scores, o_scores, (size_t)n * 4, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpyAsync(out_ids_a, o_a, (size_t)n * 8, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpyAsync(out_ids_b, o_b, (size_t)n * 8, cudaMemcpyDeviceToHost, rst));
    CU(cudaMemcpyAsync(&cnt, o_cnt, 4, cudaMemcpyDeviceToHost, rst));
    CU(cudaStreamSynchronize(rst));
    // the copies above read the other devices' lists: their buffers are freed only now
    if (cnt != (int32_t)n) return fail(SVSB_E_CUDA, "internal: pair merge returned a bad count");
    *out_count = n;
    return SVSB_OK;
}

// ------------------------------------------------------------------------------------------------
// measurement: `iters` device-resident queries through the fused path, TICKETS in flight
// ------------------------------------------------------------------------------------------------
int multi_bench_run(svsb_engine* e, const std::shared_ptr<Generation>& g, int32_t k, int32_t iters, float* total_ms, float* gemv_ms) {
    Multi* m = e->multi;
    const int64_t kk = std::min<int64_t>(k, g->n_live);
    if (kk > K_FAST_MAX) return fail(SVSB_E_INVALID, "svsb_bench_run: k <= 2048 on a multi-device engine");
    constexpr int KTIME_EVERY = 8;
    const bool ktime = gemv_ms != nullptr && g->shards[0].n_live > 0;
    CU(cudaSetDevice(root_dev(m)));
    while (ktime && m->kev.size() < (size_t)iters * 2) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); m->kev.push_back(ev); }
    cudaStream_t rst = m->kids[0]->xchg->st;
    std::vector<svsb_ticket*> ring;
    for (auto* kid : m->kids) { CU(cudaSetDevice(kid->devs[0])); CU(cudaStreamSynchronize(kid->xchg->st)); }
    CU(cudaSetDevice(root_dev(m)));
    CU(cudaEventRecord(m->ev0, rst));
    for (int it = 0; it < iters; ++it) {
        if ((int)ring.size() >= TICKETS) {            // at most TICKETS in flight: wait for the oldest
            int rc = ticket_wait(m, ring.front());
            ticket_release(m, ring.front());
            ring.erase(ring.begin());
            if (rc != SVSB_OK) return rc;
        }
        FastJob j; j.g = g.get(); j.kk = kk; j.d_q = e->bench_q.data(); j.q_off = (int64_t)(it % e->bench_nq) * e->bench_ld;
        if (ktime && it % KTIME_EVERY == 0) { j.kev0 = m->kev[2 * it]; j.kev1 = m->kev[2 * it + 1]; }
        std::unique_lock<std::mutex> lk(m->mu);
        svsb_ticket* t = free_ticket_locked(m, lk);
        if (!t) return fail(SVSB_E_STATE, "svsb_bench_run: no free ticket (pending svsb_query_submit handles?)");
        int rc = submit_locked(m, t, j, /*host_out=*/false);
        if (rc != SVSB_OK) return rc;
        ring.push_back(t);
        m->last = t;
    }
    int rc_all = SVSB_OK;
    for (auto* t : ring) { int rc = ticket_wait(m, t); ticket_release(m, t); if (rc != SVSB_OK) rc_all = rc; }
    if (rc_all != SVSB_OK) return rc_all;
    CU(cudaSetDevice(root_dev(m)));
    CU(cudaEventRecord(m->ev1, rst));
    CU(cudaEventSynchronize(m->ev1));
    float ms = 0.f; CU(cudaEventElapsedTime(&ms, m->ev0, m->ev1));
    if (total_ms) *total_ms = ms;
    if (ktime) {
        float sum = 0.f; int cnt = 0;
        for (int it = 0; it < iters; it += KTIME_EVERY) { float t = 0.f; CU(cudaEventElapsedTime(&t, m->kev[2 * it], m->kev[2 * it + 1])); sum += t; ++cnt; }
        *gemv_ms = sum * (float)iters / (float)cnt;
    } else if (gemv_ms) *gemv_ms = 0.f;
    return SVSB_OK;
}

int multi_bench_last_result(svsb_engine* e, int32_t k, float* out_scores, int64_t* out_ids, int32_t* out_count) {
    Multi* m = e->multi;
    if (!m->last) return fail(SVSB_E_STATE, "svsb_bench_last_result: no bench run yet");
    CU(cudaSetDevice(root_dev(m)));
    CU(cudaStreamSynchronize(m->kids[0]->xchg->st));
    int32_t cnt = 0;
    CU(cudaMemcpy(&cnt, m->last->d_count, 4, cudaMemcpyDeviceToHost));
    if (cnt < 0 || cnt > k) return fail(SVSB_E_INVALID, "svsb_bench_last_result: k smaller than the result");
    CU(cudaMemcpy(out_scores, m->last->d_scores, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_ids, m->last->d_ids, (size_t)cnt * 8, cudaMemcpyDeviceToHost));
    *out_count = cnt;
    return SVSB_OK;
}
