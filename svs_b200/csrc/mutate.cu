// Incremental update of the resident matrix: append + tombstone instead of the reference's full invalidate + rebuild
// after every bulk add / delete (src/svs/kb.py:1062, 1086, 1523, 1541; SURVEY.md section 8f rank 4).
//
// A generation is an immutable view (engine.cuh): rows [0, n) of a shard buffer plus an optional tombstone byte per
// row.  An update builds the NEXT view off to the side -- its own tombstone array (copy of the old one with the deleted
// ids cleared), the new rows written BEHIND the old view's last row in the same buffer (or in a grown copy when the
// buffer is full) -- and publishes it atomically.  Queries that pinned the old view never see a change.
// Row order of the live rows stays the scan order of a fresh rebuild because SQLite hands out rowids above every
// existing one (`INSERT INTO embeddings`, kb.py:557; INTEGER PRIMARY KEY, kb.py:80-83): the API checks it.
//
// svsb_apply_mutations builds and publishes in one call.  The one-process-per-GPU deployment splits the same build in
// two (svsb_shard_mutations_prepare / _commit) so that no rank publishes before every rank has built its view, and
// svsb_compact gathers the live rows of a tombstoned generation into a new buffer on the device.
#include "engine.cuh"

using namespace svsb;

namespace {

__global__ void live_init_kernel(uint8_t* __restrict__ dst, const uint8_t* __restrict__ old_live, int64_t n_old, int64_t n_new) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_new; r += step)
        dst[r] = (r < n_old && old_live) ? old_live[r] : (uint8_t)1;
}

// Every live row whose id is in the (sorted, unique) delete list dies; *found counts them.  Live ids are unique, so a
// delete id is matched by at most one row over all shards.
__global__ void tombstone_kernel(const int64_t* __restrict__ ids, uint8_t* __restrict__ live, int64_t n,
                                 const int64_t* __restrict__ del_sorted, int64_t m, unsigned long long* __restrict__ found) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += step) {
        if (!live[r]) continue;
        const int64_t id = ids[r];
        int64_t lo = 0, hi = m;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (del_sorted[mid] < id) lo = mid + 1; else hi = mid; }
        if (lo < m && del_sorted[lo] == id) { live[r] = 0; atomicAdd(found, 1ull); }
    }
}

__global__ void max_live_id_kernel(const int64_t* __restrict__ ids, const uint8_t* __restrict__ live, int64_t n, long long* __restrict__ out) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    long long best = LLONG_MIN;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += step)
        if (!live || live[r]) best = max(best, (long long)ids[r]);
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0 && best != LLONG_MIN) atomicMax(out, best);
}

// ---- compaction: scan of the tombstone bytes, then a gather of the live rows ----------------------------------------
// Block b of the scan owns rows [b * SCAN_ROWS, (b + 1) * SCAN_ROWS), 16 per thread (one 16-byte load of tombstone bytes:
// the arrays are rounded up to 16 bytes, svsb_shard_update).
constexpr int SCAN_THREADS = 256, SCAN_PER_THREAD = 16, SCAN_ROWS = SCAN_THREADS * SCAN_PER_THREAD;

// live rows among this thread's 16 (bit i of *mask: row i is live)
__device__ __forceinline__ uint32_t live_bits(const uint8_t* __restrict__ live, int64_t n, int64_t r0) {
    if (r0 >= n) return 0;
    const uint4 v = *reinterpret_cast<const uint4*>(live + r0);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t m = 0;
#pragma unroll
    for (int i = 0; i < SCAN_PER_THREAD; ++i)
        if (r0 + i < n && ((w[i >> 2] >> (8 * (i & 3))) & 0xffu)) m |= 1u << i;
    return m;
}

// exclusive prefix sum of v over the block (blockDim.x a multiple of 32, at most 1024); *total: the block's sum
__device__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {
    __shared__ uint32_t part[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
    if (lane == 31) part[w] = x;
    __syncthreads();
    if (w == 0) {
        uint32_t s = lane < nw ? part[lane] : 0;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
        part[lane] = s;
    }
    __syncthreads();
    const uint32_t excl = x - v + (w > 0 ? part[w - 1] : 0);
    *total = part[nw - 1];
    __syncthreads();                                             // part is reused by the next call
    return excl;
}

__global__ void __launch_bounds__(SCAN_THREADS) live_count_kernel(const uint8_t* __restrict__ live, int64_t n, uint32_t* __restrict__ blk) {
    const int64_t r0 = (int64_t)blockIdx.x * SCAN_ROWS + (int64_t)threadIdx.x * SCAN_PER_THREAD;
    uint32_t total;
    block_exclusive_scan(__popc(live_bits(live, n, r0)), &total);
    if (threadIdx.x == 0) blk[blockIdx.x] = total;
}

// one block: blk[0, nb) -> its exclusive prefix sums, in place
__global__ void __launch_bounds__(1024) block_offsets_kernel(uint32_t* __restrict__ blk, int64_t nb) {
    uint32_t carry = 0;
    for (int64_t c = 0; c < nb; c += blockDim.x) {
        const int64_t i = c + threadIdx.x;
        const uint32_t v = i < nb ? blk[i] : 0;
        uint32_t total;
        const uint32_t excl = block_exclusive_scan(v, &total);
        if (i < nb) blk[i] = carry + excl;
        carry += total;
    }
}

// src[j] = physical row of live row j
__global__ void __launch_bounds__(SCAN_THREADS) live_scatter_kernel(const uint8_t* __restrict__ live, int64_t n,
                                                                    const uint32_t* __restrict__ blk, uint32_t* __restrict__ src) {
    const int64_t r0 = (int64_t)blockIdx.x * SCAN_ROWS + (int64_t)threadIdx.x * SCAN_PER_THREAD;
    uint32_t m = live_bits(live, n, r0), total;
    uint32_t j = blk[blockIdx.x] + block_exclusive_scan(__popc(m), &total);
    for (; m; m &= m - 1) src[j++] = (uint32_t)(r0 + __ffs(m) - 1);
}

// one warp per destination row: row src[j] (ld floats, 16-byte loads) and its id
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ M, const int64_t* __restrict__ ids,
                                                          const uint32_t* __restrict__ src, int64_t n_out, int ld4,
                                                          float* __restrict__ dst, int64_t* __restrict__ dst_ids) {
    const int lane = threadIdx.x & 31;
    const int64_t step = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n_out; j += step) {
        const int64_t r = src[j];
        const float4* s = reinterpret_cast<const float4*>(M) + r * ld4;
        float4* o = reinterpret_cast<float4*>(dst) + j * ld4;
        for (int c = lane; c < ld4; c += 32) o[c] = __ldg(s + c);
        if (lane == 0) dst_ids[j] = ids[r];
    }
}

inline unsigned grid_for(int64_t n) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, 148 * 8)); }

struct DevTmp {                                    // frees what it handed out, on the right device
    std::vector<std::pair<int, void*>> ptrs;
    ~DevTmp() { for (auto& p : ptrs) { cudaSetDevice(p.first); cudaFree(p.second); } }
    template <class T> cudaError_t get(int dev, T** out, size_t count) {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e == cudaSuccess) { ptrs.push_back({dev, p}); *out = reinterpret_cast<T*>(p); }
        return e;
    }
};

// The load path's norm kernel over rows [0, n) of M (normalize: divide them by their norms): *max_dev / *bad are the
// statistics of the rows it saw.
int norm_pass(cudaStream_t st, int dev, float* M, int64_t n, const Generation* g, bool normalize, DevTmp& tmp, float* max_dev, int64_t* bad) {
    u64* stats = nullptr;
    CU(tmp.get(dev, &stats, 2));
    CU(cudaMemsetAsync(stats, 0, 16, st));
    CU(launch_row_norms(st, dev, M, n, g->d, g->ld, normalize ? 1 : 0, 0.001f, nullptr, stats));
    u64 h[2] = {0, 0};
    CU(cudaMemcpyAsync(h, stats, 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *max_dev = bits_f32((uint32_t)h[0]);
    *bad = (int64_t)h[1];
    return SVSB_OK;
}

// What an update asks for, checked the same way by every entry point.
struct Update {
    std::vector<int64_t> dels;                     // sorted, unique
    const float* add_rows = nullptr; const int64_t* add_ids = nullptr; int64_t n_add = 0;
};

int check_update(const char* who, const std::shared_ptr<Generation>& g, int64_t row0, const int64_t* del_ids, int64_t n_del,
                 const float* add_rows, const int64_t* add_ids, int64_t n_add, int32_t d, bool append, Update& u) {
    const std::string w(who);
    if (!g) return fail(SVSB_E_STATE, w + ": no matrix resident (rebuild)");
    if (g->ld == 0 || g->d == 0 || g->shards.empty()) return fail(SVSB_E_STATE, w + ": the resident matrix is empty (rebuild)");
    if (n_add > 0 && d != g->d) return fail(SVSB_E_STATE, w + ": row length differs from the resident matrix (rebuild)");
    for (int64_t i = 1; i < n_add; ++i)
        if (add_ids[i] <= add_ids[i - 1]) return fail(SVSB_E_STATE, w + ": inserted ids are not ascending (rebuild)");
    u.dels.assign(del_ids, del_ids + n_del);
    std::sort(u.dels.begin(), u.dels.end());
    if (std::adjacent_find(u.dels.begin(), u.dels.end()) != u.dels.end()) return fail(SVSB_E_STATE, w + ": duplicate delete id (rebuild)");
    if (append && g->n + n_add + row0 > 0xfffffff0ll) return fail(SVSB_E_STATE, w + ": more than 2^32 rows");
    u.add_rows = add_rows; u.add_ids = add_ids; u.n_add = n_add;
    return SVSB_OK;
}

// The next view of g: the deletes of u tombstoned and, when `append`, u's rows appended behind the last row of the scan
// order (the last shard).  Nothing is published.  *found: delete ids that hit a live row; *max_live: the largest live id
// after the deletes (LLONG_MIN: none), over all shards -- computed when want_max.  accept(found, max_live) runs before the
// append: a non-zero return refuses the update with that status.
template <class Accept>
int build_next(svsb_engine* e, const std::shared_ptr<Generation>& g, const Update& u, bool append, bool want_max, Accept accept,
               std::shared_ptr<Generation>& out, int64_t* found, int64_t* max_live_out) {
    const int64_t n_del = (int64_t)u.dels.size(), n_add = append ? u.n_add : 0;
    std::shared_ptr<Generation> ng(new Generation());
    ng->d = g->d; ng->ld = g->ld; ng->norm_mode = g->norm_mode; ng->max_dev = g->max_dev; ng->n_out_of_tol = g->n_out_of_tol;
    ng->shards = g->shards;
    for (auto& s : ng->shards) s.live = nullptr;               // never share (or free) the old view's arrays
    const size_t ns = ng->shards.size();
    const size_t last = ns - 1;                                  // rows are appended behind the last row of the scan order
    const bool need_live = n_del > 0 || g->has_tombstones();
    DevTmp tmp;
    std::vector<unsigned long long*> d_found(ns, nullptr);
    std::vector<long long*> d_max(ns, nullptr);
    for (size_t i = 0; i < ns; ++i) {
        Shard& s = ng->shards[i];
        const Shard& os = g->shards[i];
        const int64_t new_n = os.n + (i == last ? n_add : 0);
        CU(cudaSetDevice(s.dev));
        cudaStream_t st = e->copy_st[i];
        CU(tmp.get(s.dev, &d_found[i], 1));
        CU(tmp.get(s.dev, &d_max[i], 1));
        CU(cudaMemsetAsync(d_found[i], 0, 8, st));
        const long long lowest = LLONG_MIN;
        CU(cudaMemcpyAsync(d_max[i], &lowest, 8, cudaMemcpyHostToDevice, st));
        if (need_live && new_n > 0) {
            // owned by ng from here on (freed with it on any error below); rounded up to 16 bytes because the int8 filter
            // and the compaction scan read tombstone bytes in 16-byte units (gemv8_tma_kernel, live_bits)
            CU(cudaMalloc(&s.live, ((size_t)new_n + 15) & ~(size_t)15));
            live_init_kernel<<<grid_for(new_n), 256, 0, st>>>(s.live, os.live, os.n, new_n);
            count_launch();
            if (n_del > 0 && os.n > 0) {
                int64_t* d_del = nullptr;
                CU(tmp.get(s.dev, &d_del, (size_t)n_del));
                CU(cudaMemcpyAsync(d_del, u.dels.data(), (size_t)n_del * 8, cudaMemcpyHostToDevice, st));
                tombstone_kernel<<<grid_for(os.n), 256, 0, st>>>(os.ids, s.live, os.n, d_del, n_del, d_found[i]);
                count_launch();
            }
        }
        if (want_max && os.n > 0) {                              // largest live id after the deletes: new ids must exceed it
            max_live_id_kernel<<<grid_for(os.n), 256, 0, st>>>(os.ids, s.live, os.n, d_max[i]);
            count_launch();
        }
        CU(cudaGetLastError());
    }
    int64_t found_total = 0;
    long long max_live = LLONG_MIN;
    for (size_t i = 0; i < ns; ++i) {
        Shard& s = ng->shards[i];
        CU(cudaSetDevice(s.dev));
        unsigned long long f = 0; long long mx = LLONG_MIN;
        CU(cudaMemcpyAsync(&f, d_found[i], 8, cudaMemcpyDeviceToHost, e->copy_st[i]));
        CU(cudaMemcpyAsync(&mx, d_max[i], 8, cudaMemcpyDeviceToHost, e->copy_st[i]));
        CU(cudaStreamSynchronize(e->copy_st[i]));
        s.n_live = g->shards[i].n_live - (int64_t)f;
        found_total += (int64_t)f;
        max_live = std::max(max_live, mx);
    }
    *found = found_total;
    *max_live_out = (int64_t)max_live;
    int rc = accept(found_total, (int64_t)max_live);
    if (rc != SVSB_OK) return rc;

    if (n_add > 0) {
        Shard& s = ng->shards[last];
        const Shard& os = g->shards[last];
        const int64_t new_n = os.n + n_add;
        CU(cudaSetDevice(s.dev));
        cudaStream_t st = e->copy_st[last];
        if (!s.buf || new_n > s.buf->cap_rows) {
            // grow geometrically: one device-to-device copy now, room for further appends without one
            std::shared_ptr<ShardBuf> nb(new ShardBuf());
            nb->dev = s.dev;
            nb->cap_rows = new_n + std::max<int64_t>(new_n / 8, 1024);
            CU(cudaMalloc(&nb->M, (size_t)nb->cap_rows * ng->ld * 4));
            CU(cudaMalloc(&nb->ids, (size_t)nb->cap_rows * 8));
            if (os.n > 0) {
                CU(cudaMemcpyAsync(nb->M, os.M, (size_t)os.n * ng->ld * 4, cudaMemcpyDeviceToDevice, st));
                CU(cudaMemcpyAsync(nb->ids, os.ids, (size_t)os.n * 8, cudaMemcpyDeviceToDevice, st));
            }
            s.buf = nb; s.M = nb->M; s.ids = nb->ids;
        }
        float* dst = s.M + os.n * (int64_t)ng->ld;
        if (ng->ld == ng->d)
            CU(cudaMemcpyAsync(dst, u.add_rows, (size_t)n_add * ng->d * 4, cudaMemcpyHostToDevice, st));
        else {
            CU(cudaMemsetAsync(dst, 0, (size_t)n_add * ng->ld * 4, st));
            CU(cudaMemcpy2DAsync(dst, (size_t)ng->ld * 4, u.add_rows, (size_t)ng->d * 4, (size_t)ng->d * 4, (size_t)n_add, cudaMemcpyHostToDevice, st));
        }
        CU(cudaMemcpyAsync(s.ids + os.n, u.add_ids, (size_t)n_add * 8, cudaMemcpyHostToDevice, st));
        // the load path's norm kernel on the new rows: same policy (check / normalise), statistics folded in
        float md = 0.f; int64_t bad = 0;
        if ((rc = norm_pass(st, s.dev, dst, n_add, ng.get(), ng->norm_mode == SVSB_NORM_NORMALIZE, tmp, &md, &bad)) != SVSB_OK) return rc;
        if (ng->norm_mode != SVSB_NORM_NORMALIZE) {
            if (md > ng->max_dev || md != md) ng->max_dev = md;
            ng->n_out_of_tol += bad;
        }
        s.n = new_n;
        s.n_live += n_add;
        void* m16 = nullptr;                                     // a shadow of this buffer: convert the new rows only
        if ((rc = shadow_sync(s, ng->ld, os.n, 0, st, &m16)) != SVSB_OK) return rc;
    }
    ng->n = 0; ng->n_live = 0;
    for (auto& s : ng->shards) { ng->n += s.n; ng->n_live += s.n_live; }
    out = ng;
    return SVSB_OK;
}

}  // namespace

extern "C" int svsb_generation_rows(svsb_t* e, int64_t* physical, int64_t* live) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "no matrix resident");
    if (physical) *physical = g->n;
    if (live) *live = g->n_live;
    return SVSB_OK;
}

extern "C" int svsb_snapshot_rows(svsb_snap_t* s, int64_t* physical, int64_t* live) {
    if (!s || !s->gen) return fail(SVSB_E_INVALID, "snapshot is NULL");
    if (physical) *physical = s->gen->n;
    if (live) *live = s->gen->n_live;
    return SVSB_OK;
}

static int update_args(const char* who, const int64_t* del_ids, int64_t n_del, const float* add_rows, const int64_t* add_ids, int64_t n_add) {
    if (n_del < 0 || n_add < 0 || (n_del > 0 && !del_ids) || (n_add > 0 && (!add_rows || !add_ids)))
        return fail(SVSB_E_INVALID, std::string(who) + ": bad arguments");
    return SVSB_OK;
}

// loads, updates and compactions wait for a prepared update to be committed or dropped
static int busy(const svsb_engine* e, const char* who) {
    if (e->loading) return fail(SVSB_E_STATE, std::string(who) + ": a load is in progress");
    if (e->has_pending) return fail(SVSB_E_STATE, std::string(who) + ": a prepared update is pending (svsb_shard_mutations_commit)");
    return SVSB_OK;
}

extern "C" int svsb_apply_mutations(svsb_t* e, const int64_t* del_ids, int64_t n_del, const float* add_rows, const int64_t* add_ids,
                                    int64_t n_add, int32_t d, uint64_t* generation) {
    static const char* who = "svsb_apply_mutations";
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    int rc = update_args(who, del_ids, n_del, add_rows, add_ids, n_add);
    if (rc != SVSB_OK) return rc;
    std::lock_guard<std::mutex> mlk(e->mutate_mu);
    if ((rc = busy(e, who)) != SVSB_OK) return rc;
    auto g = pin(e);
    Update u;
    if ((rc = check_update(who, g, e->shard_row0, del_ids, n_del, add_rows, add_ids, n_add, d, true, u)) != SVSB_OK) return rc;
    std::shared_ptr<Generation> ng;
    int64_t found = 0, max_live = 0;
    rc = build_next(e, g, u, true, n_add > 0, [&](int64_t f, int64_t mx) -> int {
        if (f != n_del) {
            char buf[160];
            snprintf(buf, sizeof buf, "svsb_apply_mutations: %lld of %lld deleted ids are not live rows of the resident matrix (rebuild)",
                     (long long)(n_del - f), (long long)n_del);
            return fail(SVSB_E_STATE, buf);
        }
        if (n_add > 0 && mx != LLONG_MIN && add_ids[0] <= mx)
            return fail(SVSB_E_STATE, "svsb_apply_mutations: an inserted id is not above every live id (rebuild)");
        return SVSB_OK;
    }, ng, &found, &max_live);
    if (rc != SVSB_OK) return rc;
    // the update is relative to generation g: if a load (or an invalidate) replaced it meanwhile, publishing this view would
    // resurrect the old table -- refuse, the caller rebuilds
    if (pin(e) != g) return fail(SVSB_E_STATE, "svsb_apply_mutations: the resident generation changed during the update (rebuild)");
    return publish_generation(e, ng, generation);
}

extern "C" int svsb_shard_mutations_prepare(svsb_t* e, const int64_t* del_ids, int64_t n_del, const float* add_rows, const int64_t* add_ids,
                                            int64_t n_add, int32_t d, int32_t append_here, int64_t* found, int64_t* max_live_id) {
    static const char* who = "svsb_shard_mutations_prepare";
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (!found || !max_live_id) return fail(SVSB_E_INVALID, "svsb_shard_mutations_prepare: NULL output");
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, "svsb_shard_mutations_prepare: a sharded engine owns exactly one device");
    int rc = update_args(who, del_ids, n_del, add_rows, add_ids, n_add);
    if (rc != SVSB_OK) return rc;
    std::lock_guard<std::mutex> mlk(e->mutate_mu);
    if ((rc = busy(e, who)) != SVSB_OK) return rc;
    auto g = pin(e);
    Update u;
    if ((rc = check_update(who, g, e->shard_row0, del_ids, n_del, add_rows, add_ids, n_add, d, append_here != 0, u)) != SVSB_OK) return rc;
    std::shared_ptr<Generation> ng;
    if ((rc = build_next(e, g, u, append_here != 0, true, [](int64_t, int64_t) -> int { return SVSB_OK; }, ng, found, max_live_id)) != SVSB_OK)
        return rc;
    // everything that can fail happens here: the commit only swaps pointers
    if ((rc = filter_attach(e, ng.get())) != SVSB_OK) return rc;
    std::lock_guard<std::mutex> lk(e->mu);
    if (e->current != g) return fail(SVSB_E_STATE, "svsb_shard_mutations_prepare: the resident generation changed during the update");
    e->pending = ng;
    e->has_pending = true;
    return SVSB_OK;
}

extern "C" int svsb_shard_mutations_commit(svsb_t* e, int32_t publish, uint64_t* generation) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    std::shared_ptr<Generation> ng;                               // a dropped generation is freed outside the lock
    std::lock_guard<std::mutex> mlk(e->mutate_mu);
    std::lock_guard<std::mutex> lk(e->mu);
    ng.swap(e->pending);
    e->has_pending = false;
    if (!publish) return SVSB_OK;
    if (!ng) return fail(SVSB_E_STATE, "svsb_shard_mutations_commit: no update is prepared");
    ng->id = e->next_gen++;
    e->current = ng;
    if (generation) *generation = ng->id;
    return SVSB_OK;
}

extern "C" int svsb_compact(svsb_t* e, int64_t global_row0, uint64_t* generation) {
    static const char* who = "svsb_compact";
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (global_row0 < 0) return fail(SVSB_E_INVALID, "svsb_compact: negative row offset");
    if (e->devs.size() != 1) return fail(SVSB_E_INVALID, "svsb_compact: a multi-device engine compacts by reloading");
    std::lock_guard<std::mutex> mlk(e->mutate_mu);
    int rc = busy(e, who);
    if (rc != SVSB_OK) return rc;
    auto g = pin(e);
    if (!g) return fail(SVSB_E_NOT_LOADED, "svsb_compact: no matrix resident");
    if (g->n_live + global_row0 > 0xfffffff0ll) return fail(SVSB_E_INVALID, "svsb_compact: more than 2^32 rows in total are not supported");
    const Shard& os = g->shards[0];
    std::shared_ptr<Generation> ng(new Generation());
    ng->d = g->d; ng->ld = g->ld; ng->norm_mode = g->norm_mode; ng->max_dev = g->max_dev; ng->n_out_of_tol = g->n_out_of_tol;
    ng->n = ng->n_live = g->n_live;
    Shard s;
    s.dev = os.dev; s.row0 = global_row0; s.n = s.n_live = g->n_live;
    if (!g->has_tombstones()) {                                   // every row is live: the same buffers at the new offset
        s.buf = os.buf; s.M = os.M; s.ids = os.ids;
    } else if (s.n > 0) {
        CU(cudaSetDevice(s.dev));
        cudaStream_t st = e->copy_st[0];
        std::shared_ptr<ShardBuf> nb(new ShardBuf());             // a load's buffer for n_live rows (alloc_generation)
        nb->dev = s.dev;
        nb->cap_rows = shard_capacity(s.n);
        CU(cudaMalloc(&nb->M, (size_t)nb->cap_rows * g->ld * 4));
        CU(cudaMalloc(&nb->ids, (size_t)nb->cap_rows * 8));
        DevTmp tmp;
        const int64_t nb_scan = (os.n + SCAN_ROWS - 1) / SCAN_ROWS;
        uint32_t *blk = nullptr, *src = nullptr;
        CU(tmp.get(s.dev, &blk, (size_t)nb_scan));
        CU(tmp.get(s.dev, &src, (size_t)s.n));
        live_count_kernel<<<(unsigned)nb_scan, SCAN_THREADS, 0, st>>>(os.live, os.n, blk);
        block_offsets_kernel<<<1, 1024, 0, st>>>(blk, nb_scan);
        live_scatter_kernel<<<(unsigned)nb_scan, SCAN_THREADS, 0, st>>>(os.live, os.n, blk, src);
        gather_rows_kernel<<<(unsigned)std::min<int64_t>((s.n + 7) / 8, 148 * 16), 256, 0, st>>>(os.M, os.ids, src, s.n, g->ld / 4, nb->M, nb->ids);
        for (int i = 0; i < 4; ++i) count_launch();
        CU(cudaGetLastError());
        s.buf = nb; s.M = nb->M; s.ids = nb->ids;
        // the statistics of a fresh load of these rows; normalised rows keep the old ones (their rows' superset's: conservative)
        if (g->norm_mode != SVSB_NORM_NORMALIZE) {
            float md = 0.f; int64_t bad = 0;
            if ((rc = norm_pass(st, s.dev, s.M, s.n, g.get(), false, tmp, &md, &bad)) != SVSB_OK) return rc;
            ng->max_dev = md; ng->n_out_of_tol = bad;
        }
        CU(cudaStreamSynchronize(st));
    } else if (g->norm_mode != SVSB_NORM_NORMALIZE) {
        ng->max_dev = 0.f; ng->n_out_of_tol = 0;                  // a load of no rows
    }
    ng->shards.push_back(s);
    if ((rc = publish_generation(e, ng, generation)) != SVSB_OK) return rc;   // builds the filters' shadows as a load does
    std::lock_guard<std::mutex> lk(e->mu);
    e->shard_row0 = global_row0;
    return SVSB_OK;
}
