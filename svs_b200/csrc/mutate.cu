// Incremental update of the resident matrix: append + tombstone instead of the reference's full invalidate + rebuild
// after every bulk add / delete (src/svs/kb.py:1062, 1086, 1523, 1541; SURVEY.md section 8f rank 4).
//
// A generation is an immutable view (engine.cuh): rows [0, n) of a shard buffer plus an optional tombstone byte per
// row.  svsb_apply_mutations builds the NEXT view off to the side -- its own tombstone array (copy of the old one with
// the deleted ids cleared), the new rows written BEHIND the old view's last row in the same buffer (or in a grown copy
// when the buffer is full) -- and publishes it atomically.  Queries that pinned the old view never see a change.
// Row order of the live rows stays the scan order of a fresh rebuild because SQLite hands out rowids above every
// existing one (`INSERT INTO embeddings`, kb.py:557; INTEGER PRIMARY KEY, kb.py:80-83): the API checks it.
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

extern "C" int svsb_apply_mutations(svsb_t* e, const int64_t* del_ids, int64_t n_del, const float* add_rows, const int64_t* add_ids,
                                    int64_t n_add, int32_t d, uint64_t* generation) {
    if (!e) return fail(SVSB_E_INVALID, "engine is NULL");
    if (n_del < 0 || n_add < 0 || (n_del > 0 && !del_ids) || (n_add > 0 && (!add_rows || !add_ids)))
        return fail(SVSB_E_INVALID, "svsb_apply_mutations: bad arguments");
    std::lock_guard<std::mutex> mlk(e->mutate_mu);
    if (e->loading) return fail(SVSB_E_STATE, "svsb_apply_mutations: a load is in progress");
    auto g = pin(e);
    if (!g) return fail(SVSB_E_STATE, "svsb_apply_mutations: no matrix resident (rebuild)");
    if (g->ld == 0 || g->d == 0 || g->shards.empty()) return fail(SVSB_E_STATE, "svsb_apply_mutations: the resident matrix is empty (rebuild)");
    if (n_add > 0 && d != g->d) return fail(SVSB_E_STATE, "svsb_apply_mutations: row length differs from the resident matrix (rebuild)");
    for (int64_t i = 1; i < n_add; ++i)
        if (add_ids[i] <= add_ids[i - 1]) return fail(SVSB_E_STATE, "svsb_apply_mutations: inserted ids are not ascending (rebuild)");
    std::vector<int64_t> dels(del_ids, del_ids + n_del);
    std::sort(dels.begin(), dels.end());
    if (std::adjacent_find(dels.begin(), dels.end()) != dels.end()) return fail(SVSB_E_STATE, "svsb_apply_mutations: duplicate delete id (rebuild)");
    if (g->n + n_add + e->shard_row0 > 0xfffffff0ll) return fail(SVSB_E_STATE, "svsb_apply_mutations: more than 2^32 rows");

    // the next view: same buffers, its own tombstone arrays
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
            // copies a partial last tile's tombstone bytes in 16-byte units (gemv8_tma_kernel)
            CU(cudaMalloc(&s.live, ((size_t)new_n + 15) & ~(size_t)15));
            live_init_kernel<<<grid_for(new_n), 256, 0, st>>>(s.live, os.live, os.n, new_n);
            count_launch();
            if (n_del > 0 && os.n > 0) {
                int64_t* d_del = nullptr;
                CU(tmp.get(s.dev, &d_del, (size_t)n_del));
                CU(cudaMemcpyAsync(d_del, dels.data(), (size_t)n_del * 8, cudaMemcpyHostToDevice, st));
                tombstone_kernel<<<grid_for(os.n), 256, 0, st>>>(os.ids, s.live, os.n, d_del, n_del, d_found[i]);
                count_launch();
            }
        }
        if (n_add > 0 && os.n > 0) {                              // largest live id after the deletes: new ids must exceed it
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
    if (found_total != n_del) {
        char buf[160];
        snprintf(buf, sizeof buf, "svsb_apply_mutations: %lld of %lld deleted ids are not live rows of the resident matrix (rebuild)",
                 (long long)(n_del - found_total), (long long)n_del);
        return fail(SVSB_E_STATE, buf);
    }
    if (n_add > 0 && max_live != LLONG_MIN && add_ids[0] <= max_live)
        return fail(SVSB_E_STATE, "svsb_apply_mutations: an inserted id is not above every live id (rebuild)");

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
            CU(cudaMemcpyAsync(dst, add_rows, (size_t)n_add * ng->d * 4, cudaMemcpyHostToDevice, st));
        else {
            CU(cudaMemsetAsync(dst, 0, (size_t)n_add * ng->ld * 4, st));
            CU(cudaMemcpy2DAsync(dst, (size_t)ng->ld * 4, add_rows, (size_t)ng->d * 4, (size_t)ng->d * 4, (size_t)n_add, cudaMemcpyHostToDevice, st));
        }
        CU(cudaMemcpyAsync(s.ids + os.n, add_ids, (size_t)n_add * 8, cudaMemcpyHostToDevice, st));
        // the load path's norm kernel on the new rows: same policy (check / normalise), statistics folded in
        u64* stats = nullptr;
        CU(tmp.get(s.dev, &stats, 2));
        CU(cudaMemsetAsync(stats, 0, 16, st));
        CU(launch_row_norms(st, s.dev, dst, n_add, ng->d, ng->ld, ng->norm_mode == SVSB_NORM_NORMALIZE ? 1 : 0, 0.001f, nullptr, stats));
        u64 h[2] = {0, 0};
        CU(cudaMemcpyAsync(h, stats, 16, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        const float md = bits_f32((uint32_t)h[0]);
        if (ng->norm_mode != SVSB_NORM_NORMALIZE) {
            if (md > ng->max_dev || md != md) ng->max_dev = md;
            ng->n_out_of_tol += (int64_t)h[1];
        }
        s.n = new_n;
        s.n_live += n_add;
        void* m16 = nullptr;                                     // a shadow of this buffer: convert the new rows only
        int rc = shadow_sync(s, ng->ld, os.n, 0, st, &m16);
        if (rc != SVSB_OK) return rc;
    }
    ng->n = 0; ng->n_live = 0;
    for (auto& s : ng->shards) { ng->n += s.n; ng->n_live += s.n_live; }
    // the update is relative to generation g: if a load (or an invalidate) replaced it meanwhile, publishing this view would
    // resurrect the old table -- refuse, the caller rebuilds
    if (pin(e) != g) return fail(SVSB_E_STATE, "svsb_apply_mutations: the resident generation changed during the update (rebuild)");
    return publish_generation(e, ng, generation);
}
