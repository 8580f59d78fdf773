// K3/K4 -- exact top-k over the fp32 scores, plus the cross-shard candidate merge (K5's compute half).
//
// Replaces get_top_k (reference src/svs/util.py:190-203: np.argpartition + sorted) and the
// `emb_id_lookup[index]` gather (src/svs/kb.py:1188, 1626).
//
// Scheme ("group maxima + exact refilter"), all in ONE single-CTA kernel after the GEMV:
//   The GEMV leaves, next to scores[n], the maximum KEY of every group of m = 2^shift consecutive rows
//   (G = ceil(n/m) <= 16384 entries).  Let tau be the k-th largest group maximum.  There are k distinct
//   rows with key >= tau, so tau is a lower bound on the k-th largest key overall, and every row with
//   key >= tau lives in one of the k groups whose maximum is >= tau.  The kernel therefore
//     1. finds tau among the G group maxima (range-adaptive radix select in shared memory),
//     2. rescans only those k groups (k*m scores, not n) and collects the rows with key >= tau
//        (typically k + a handful; never more than k*m),
//     3. selects/sorts the candidates exactly (bitonic sort in shared memory), and
//     4. writes (score, embeddings.id) pairs, resetting the group maxima for the next query.
//   Keys are unique per row (common.cuh), so the result is the exact top-k under the order
//   (score desc, row asc) whatever the data looks like -- ties, sorted input, NaNs included.
//   Work: ONE pass over G*8 bytes (into shared memory; everything after that is on-chip) + k*m*4 bytes of
//   scores, all L2 hits; no pass over the n scores.  Three dependent global round trips in total.
//
// k > K_FAST_MAX (e.g. the notebooks' n = len(kb) full ranking) takes a plain global bitonic sort.
#include "select_common.cuh"

#include <algorithm>

namespace svsb {

// kk-th largest (1-based) of keys[0..count), count >= kk >= 1.  All threads of the block call it and
// all receive the result.  keys may be in global or shared memory.  Uses sm.hist / sm.sortbuf.
// have_range: sm.bcast64[0..1] already hold min / max of the keys (saves a pass).
__device__ u64 block_kth_largest(const u64* keys, int64_t count, int kk, SelectSmem& sm, bool have_range = false) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    if (!have_range) {
        // pass 0: range of the keys
        u64 mn = ~0ull, mx = 0ull;
        for (int64_t i = tid; i < count; i += blockDim.x) { const u64 v = keys[i]; mn = v < mn ? v : mn; mx = v > mx ? v : mx; }
        mn = warp_min_u64(mn); mx = warp_max_u64(mx);
        if (lane == 0) { sm.red_a[warp] = mn; sm.red_b[warp] = mx; }
        __syncthreads();
        if (warp == 0) {
            mn = lane < nwarps ? sm.red_a[lane] : ~0ull;
            mx = lane < nwarps ? sm.red_b[lane] : 0ull;
            mn = warp_min_u64(mn); mx = warp_max_u64(mx);
            if (lane == 0) { sm.bcast64[0] = mn; sm.bcast64[1] = mx; }
        }
        __syncthreads();
    }
    u64 lo = sm.bcast64[0], hi = sm.bcast64[1];
    int remaining = kk;
    __syncthreads();

    while (true) {
        const int shift = max(0, bitlen64(hi - lo) - HIST_BITS);
        for (int i = tid; i < HIST_BINS; i += blockDim.x) sm.hist[i] = 0;
        __syncthreads();
        for (int64_t i = tid; i < count; i += blockDim.x) {
            const u64 v = keys[i];
            if (v >= lo && v <= hi) atomicAdd(&sm.hist[(uint32_t)((v - lo) >> shift)], 1u);
        }
        __syncthreads();
        // Find, from the top, the bin where the cumulative count reaches `remaining`.
        // Level 1: 32 chunks of 64 bins, chunk c = bins [64c, 64c+64); each warp sums chunks (conflict-free).
        for (int cidx = warp; cidx < 32; cidx += nwarps) {
            uint32_t v = sm.hist[cidx * 64 + lane] + sm.hist[cidx * 64 + 32 + lane];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) sm.red_a[cidx] = (u64)v;
        }
        __syncthreads();
        if (warp == 0) {
            // lane l looks at chunk (31 - l): top-down inclusive prefix over chunks
            const uint32_t mysum = (uint32_t)sm.red_a[31 - lane];
            uint32_t incl = mysum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
            const uint32_t excl = incl - mysum;
            const unsigned hitmask = __ballot_sync(0xffffffffu, excl < (uint32_t)remaining && incl >= (uint32_t)remaining);
            const int src = __ffs(hitmask) - 1;                       // exactly one lane qualifies
            const int chunk = 31 - src;
            const uint32_t above_chunk = __shfl_sync(0xffffffffu, excl, src);
            // Level 2: inside the chunk, lane l looks at bins (top - l) and (top - 32 - l)
            const int top = chunk * 64 + 63;
            const uint32_t h0 = sm.hist[top - lane], h1 = sm.hist[top - 32 - lane];
            uint32_t p0 = h0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, p0, o); if (lane >= o) p0 += t; }
            const uint32_t first_half = __shfl_sync(0xffffffffu, p0, 31);
            uint32_t p1 = h1;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, p1, o); if (lane >= o) p1 += t; }
            const uint32_t need = (uint32_t)remaining - above_chunk;   // 1-based position inside the chunk
            const uint32_t e0 = p0 - h0, e1 = first_half + p1 - h1;    // exclusive prefixes (top-down)
            if (e0 < need && p0 >= need) { sm.bcast32[0] = top - lane; sm.bcast32[1] = (int)(above_chunk + e0); }
            if (e1 < need && first_half + p1 >= need) { sm.bcast32[0] = top - 32 - lane; sm.bcast32[1] = (int)(above_chunk + e1); }
        }
        __syncthreads();
        const int bin = sm.bcast32[0];
        const int above = sm.bcast32[1];
        const uint32_t inbin = sm.hist[bin];
        remaining -= above;
        const u64 nlo = lo + ((u64)bin << shift);
        u64 nhi = nlo + (((u64)1 << shift) - 1);
        if (nhi > hi || nhi < nlo) nhi = hi;
        lo = nlo; hi = nhi;
        __syncthreads();
        if (shift == 0) return lo;                          // bin holds one key value: that is the answer
        if (inbin <= (uint32_t)RANK_SORT_MAX) break;
    }
    // finish in shared memory: collect the (few) keys of the final bin, pick the remaining-th by rank
    if (tid == 0) sm.counter = 0;
    __syncthreads();
    for (int64_t i = tid; i < count; i += blockDim.x) {
        const u64 v = keys[i];
        if (v >= lo && v <= hi) { const uint32_t p = atomicAdd(&sm.counter, 1u); if (p < (uint32_t)RANK_SORT_MAX) sm.sortbuf[p] = v; }
    }
    __syncthreads();
    const int c = (int)min(sm.counter, (uint32_t)RANK_SORT_MAX);
    if (tid < c) {
        const u64 mine = sm.sortbuf[tid];
        int rank = 0;
        for (int j = 0; j < c; ++j) rank += (sm.sortbuf[j] > mine) ? 1 : 0;
        if (rank == remaining - 1) sm.bcast64[0] = mine;
    }
    __syncthreads();
    const u64 ans = sm.bcast64[0];
    __syncthreads();
    return ans;
}

// ---------------------------------------------------------------------------------------------
// Peer exchange helpers.  Publication: every thread has stored its part of the record into the peers' windows;
// after the CTA barrier thread p stores the count, fences at system scope (cumulative over the barrier) and
// release-stores the sequence number into rank p's flag.  The consumer acquires the flag before reading.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void peer_publish(const PeerPush& push, int count) {
    __syncthreads();
    const int p = threadIdx.x;
    if (p < push.world) {
        push.rec[p][2 * push.cap] = (u64)(uint32_t)count;
        __threadfence_system();
        st_release_sys(push.flag[p], push.seq);
    }
}

// Query upload without the copy engine: one small CTA reads the query from pinned (mapped) host memory over PCIe and
// writes it to HBM, so the synchronous peer path is kernels only (no copy-engine -> compute hand-off before the
// similarity pass).  ld.cv: never serve host memory the CPU rewrites per query from a stale cache line.
__global__ void __launch_bounds__(256) stage_query_kernel(const float4* __restrict__ host_q, float4* __restrict__ d_q, int ld4) {
    pdl_trigger();                                 // the similarity kernel may start streaming the matrix right away
    for (int c = threadIdx.x; c < ld4; c += blockDim.x) {
        float4 v;
        asm volatile("ld.global.cv.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(host_q + c));
        d_q[c] = v;
    }
}

cudaError_t launch_stage_query(cudaStream_t st, const float* host_q_mapped, float* d_q, int ld)
{
    if (ld <= 0 || (ld & 3)) return cudaErrorInvalidValue;
    // never itself a programmatic dependent: it overwrites the query buffer the previous call's kernels read
    stage_query_kernel<<<1, 256, 0, st>>>(reinterpret_cast<const float4*>(host_q_mapped), reinterpret_cast<float4*>(d_q), ld / 4);
    count_launch();
    return cudaGetLastError();
}

__global__ void __launch_bounds__(32) push_empty_kernel(const __grid_constant__ PeerPush push) { peer_publish(push, 0); }

cudaError_t launch_push_empty(cudaStream_t st, const PeerPush& push)
{
    if (push.world < 1 || push.world > XCHG_MAX_RANKS) return cudaErrorInvalidValue;
    push_empty_kernel<<<1, 32, 0, st>>>(push);
    count_launch();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// The selection kernel (one CTA).
// ---------------------------------------------------------------------------------------------
constexpr int SEL_KEYS_CAP = (int)GROUPS_TARGET;     // group maxima staged in shared memory
constexpr int SEL_KEYS_PER_THREAD = SEL_KEYS_CAP / SEL_THREADS;   // 16

struct SelectKeysSmem {
    SelectSmem base;
    u64 keys[SEL_KEYS_CAP];
    uint32_t hits[K_FAST_MAX];
};

__global__ void __launch_bounds__(SEL_THREADS, 1)
select_topk_kernel(const float* __restrict__ scores, int64_t n, u64* gmax, int group_shift,
                   int k, const int64_t* __restrict__ ids, int64_t row0, u64* cand, int64_t cand_cap,
                   u64* __restrict__ out_keys, float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                   int32_t* __restrict__ out_count, u64* __restrict__ dbg, const __grid_constant__ PeerPush push,
                   const SelectStrides bs)
{
    extern __shared__ __align__(16) unsigned char sel_smem_raw[];
    SelectKeysSmem& big = *reinterpret_cast<SelectKeysSmem*>(sel_smem_raw);
    {   // one CTA per query of a batch (grid 1, all strides 0: the single query)
        const int64_t qi = blockIdx.x;
        scores += qi * bs.scores; gmax += qi * bs.gmax; cand += qi * bs.cand;
        out_keys += qi * bs.keys; out_scores += qi * bs.oscores; out_ids += qi * bs.ids; out_count += qi * bs.count;
    }
#define SEL_STAMP(i) do { if (dbg && threadIdx.x == 0) { u64 t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); dbg[i] = t_; } } while (0)
    pdl_wait();                                    // scores and group maxima come from the similarity kernel
    pdl_trigger();
    SEL_STAMP(0);
    SelectSmem& sm = big.base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int kk = (int)min((int64_t)k, n);
    const int G = (int)((n + ((int64_t)1 << group_shift) - 1) >> group_shift);    // <= SEL_KEYS_CAP
    const int m = 1 << group_shift;

    // 1. one pass over the group maxima: global -> registers (independent loads) -> shared; reset them;
    //    min / max on the way
    {
        u64 r[SEL_KEYS_PER_THREAD];
#pragma unroll
        for (int j = 0; j < SEL_KEYS_PER_THREAD; ++j) { const int i = tid + j * SEL_THREADS; r[j] = i < G ? gmax[i] : 0ull; }
        u64 mn = ~0ull, mx = 0ull;
#pragma unroll
        for (int j = 0; j < SEL_KEYS_PER_THREAD; ++j) {
            const int i = tid + j * SEL_THREADS;
            if (i < G) { big.keys[i] = r[j]; gmax[i] = 0ull; mn = r[j] < mn ? r[j] : mn; mx = r[j] > mx ? r[j] : mx; }
        }
        mn = warp_min_u64(mn); mx = warp_max_u64(mx);
        if (lane == 0) { sm.red_a[warp] = mn; sm.red_b[warp] = mx; }
        if (tid == 0) sm.counter = 0;
        __syncthreads();
        if (warp == 0) {
            mn = lane < nwarps ? sm.red_a[lane] : ~0ull;
            mx = lane < nwarps ? sm.red_b[lane] : 0ull;
            mn = warp_min_u64(mn); mx = warp_max_u64(mx);
            if (lane == 0) { sm.bcast64[0] = mn; sm.bcast64[1] = mx; }
        }
        __syncthreads();
    }

    SEL_STAMP(1);
    // 2. threshold: the kk-th largest group maximum (0 = "every group" when there are <= kk groups)
    u64 tau = 0;
    if (G > kk) tau = block_kth_largest(big.keys, G, kk, sm, /*have_range=*/true);
    SEL_STAMP(2);

    // 3. the groups whose maximum reaches tau (exactly kk of them, or all G)
    if (tid == 0) sm.counter = 0;
    __syncthreads();
    for (int i = tid; i < G; i += SEL_THREADS)
        if (big.keys[i] >= tau) { const uint32_t p = atomicAdd(&sm.counter, 1u); if (p < (uint32_t)K_FAST_MAX) big.hits[p] = (uint32_t)i; }
    __syncthreads();
    const int nhits = (int)min(sm.counter, (uint32_t)K_FAST_MAX);
    __syncthreads();
    SEL_STAMP(3);

    // 4. candidates: rows of those groups with key >= tau (flattened: independent, coalesced loads).
    //    The first SORT_CAP go straight into the sort buffer; any overflow goes to `cand` in global memory.
    if (tid == 0) sm.counter = 0;
    __syncthreads();
    const int64_t items = (int64_t)nhits << group_shift;
    constexpr int CB = 8;                                   // loads in flight per thread
    for (int64_t it0 = tid; it0 < items; it0 += (int64_t)SEL_THREADS * CB) {
        int64_t rr[CB]; float sc[CB];
#pragma unroll
        for (int u = 0; u < CB; ++u) {
            const int64_t it = it0 + (int64_t)u * SEL_THREADS;
            rr[u] = -1;
            if (it < items) {
                const int64_t r = ((int64_t)big.hits[it >> group_shift] << group_shift) + (it & (m - 1));
                if (r < n) rr[u] = r;
            }
        }
#pragma unroll
        for (int u = 0; u < CB; ++u) sc[u] = rr[u] >= 0 ? scores[rr[u]] : 0.f;
#pragma unroll
        for (int u = 0; u < CB; ++u) {
            if (rr[u] < 0) continue;
            const u64 key = make_key(sc[u], (uint32_t)rr[u]);
            if (key >= tau) {
                const uint32_t p = atomicAdd(&sm.counter, 1u);
                if (p < (uint32_t)SORT_CAP) sm.sortbuf[p] = key;
                else if ((int64_t)(p - SORT_CAP) < cand_cap) cand[p - SORT_CAP] = key;
            }
        }
    }
    __syncthreads();
    const int64_t C = (int64_t)sm.counter;
    __syncthreads();
    SEL_STAMP(4);
    if (dbg && tid == 0) { dbg[8] = (u64)C; dbg[9] = (u64)nhits; }

    // 5. exact top-kk of the candidates, sorted
    if (C > SORT_CAP) {
        // rare (adversarial order / massive ties): move everything to `cand`, second-level select there
        const int64_t over = min(C - SORT_CAP, cand_cap - SORT_CAP);
        for (int i = tid; i < SORT_CAP; i += SEL_THREADS) cand[over + i] = sm.sortbuf[i];
        __syncthreads();
        const int64_t total = over + SORT_CAP;
        const u64 tau2 = block_kth_largest(cand, total, kk, sm);
        if (tid == 0) sm.counter = 0;
        __syncthreads();
        for (int64_t i = tid; i < total; i += SEL_THREADS) {
            const u64 v = cand[i];
            if (v >= tau2) { const uint32_t p = atomicAdd(&sm.counter, 1u); if (p < (uint32_t)SORT_CAP) sm.sortbuf[p] = v; }
        }
        __syncthreads();
    }
    const int c = (int)min(sm.counter, (uint32_t)SORT_CAP);
    const u64* sorted = sm.sortbuf;
    if (c <= RANK_SORT_MAX) {
        u64* dst = reinterpret_cast<u64*>(sm.payload);       // unused by this kernel otherwise
        block_rank_sort_desc(sm.sortbuf, dst, c);
        sorted = dst;
    } else {
        int np2 = 1; while (np2 < c) np2 <<= 1;
        for (int i = c + tid; i < np2; i += SEL_THREADS) sm.sortbuf[i] = 0ull;
        __syncthreads();
        block_bitonic_desc<false>(sm.sortbuf, nullptr, np2);
    }
    SEL_STAMP(5);

    // 6. epilogue: (score, embeddings.id), keys re-based to global rows for the cross-shard merge
    for (int i = tid; i < kk; i += SEL_THREADS) {
        const u64 key = sorted[i];
        const uint32_t row = key_row(key);
        const int64_t grow = row0 + (int64_t)row;
        const u64 gkey = (key & 0xffffffff00000000ull) | (u64)(uint32_t)(~(uint32_t)grow);
        const int64_t id = ids ? ids[row] : grow;
        out_keys[i] = gkey;
        out_scores[i] = key_score(key);
        out_ids[i] = id;
        // the exchange step, fused: the record goes straight into every rank's gather window (peer stores)
        for (int p = 0; p < push.world; ++p) { push.rec[p][i] = gkey; push.rec[p][push.cap + i] = (u64)id; }
    }
    if (tid == 0) *out_count = kk;
    if (push.world > 0) peer_publish(push, kk);
    SEL_STAMP(6);
#undef SEL_STAMP
}

cudaError_t launch_select(cudaStream_t st, const float* scores, int64_t n, u64* gmax, int group_shift,
                          int k, const int64_t* ids, int64_t row0, u64* cand, int64_t cand_cap,
                          u64* out_keys, float* out_scores, int64_t* out_ids, int32_t* out_count, u64* dbg,
                          const PeerPush* push)
{
    if (k < 1 || k > K_FAST_MAX || n < 1) return cudaErrorInvalidValue;
    PeerPush pp{};
    if (push) { pp = *push; if (pp.world < 1 || pp.world > XCHG_MAX_RANKS || pp.cap < k) return cudaErrorInvalidValue; }
    static bool attr_set[64] = {false};
    int dev = 0; cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(select_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectKeysSmem));
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    if (((n + ((int64_t)1 << group_shift) - 1) >> group_shift) > SEL_KEYS_CAP) return cudaErrorInvalidValue;
    cudaError_t le = launch_kernel(select_topk_kernel, dim3(1), dim3(SEL_THREADS), sizeof(SelectKeysSmem), st, scores, n, gmax, group_shift, k,
                                   ids, row0, cand, cand_cap, out_keys, out_scores, out_ids, out_count, dbg, pp, SelectStrides{});
    count_launch();
    return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t launch_select_batch(cudaStream_t st, int b, const SelectStrides& bs, const float* scores, int64_t n, u64* gmax, int group_shift,
                                int k, const int64_t* ids, int64_t row0, u64* cand, int64_t cand_cap,
                                u64* out_keys, float* out_scores, int64_t* out_ids, int32_t* out_count)
{
    if (b < 1 || k < 1 || k > K_FAST_MAX || n < 1) return cudaErrorInvalidValue;
    static bool attr_set[64] = {false};
    int dev = 0; cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(select_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectKeysSmem));
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    if (((n + ((int64_t)1 << group_shift) - 1) >> group_shift) > SEL_KEYS_CAP) return cudaErrorInvalidValue;
    PeerPush none{};
    select_topk_kernel<<<b, SEL_THREADS, sizeof(SelectKeysSmem), st>>>(scores, n, gmax, group_shift, k, ids, row0, cand, cand_cap,
                                                                       out_keys, out_scores, out_ids, out_count, nullptr, none, bs);
    count_launch();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// group maxima from a score vector (selection-only entry point)
// ---------------------------------------------------------------------------------------------
__global__ void groupmax_kernel(const float* __restrict__ scores, int64_t n, u64* __restrict__ gmax, int group_shift) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t nchunks = (n + 31) / 32;                       // 32 rows per warp step; 32 | group size
    for (int64_t c = warp_global; c < nchunks; c += nwarps) {
        const int64_t r = c * 32 + lane;
        u64 key = r < n ? make_key(scores[r], (uint32_t)r) : 0ull;
        key = warp_max_u64(key);
        if (lane == 0) atomicMax(&gmax[(c * 32) >> group_shift], key);
    }
}

cudaError_t launch_groupmax(cudaStream_t st, int device, const float* scores, int64_t n, u64* gmax, int group_shift) {
    if (n <= 0) return cudaSuccess;
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count(device) * 8;
    if (blocks > cap) blocks = cap;
    groupmax_kernel<<<(unsigned)blocks, 256, 0, st>>>(scores, n, gmax, group_shift);
    count_launch();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// large-k path: sort every key (global bitonic sort, shared-memory fused inner steps)
// ---------------------------------------------------------------------------------------------
constexpr int BS_CHUNK = 2048;                                  // keys per CTA in the fused steps
constexpr int BS_THREADS = 1024;

__global__ void fs_make_keys_kernel(const float* __restrict__ scores, int64_t n, int64_t np2, u64* __restrict__ keys,
                                    u64* __restrict__ gmax, int64_t G) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < np2; i += stride) {
        keys[i] = i < n ? make_key(scores[i], (uint32_t)i) : 0ull;
        if (i < G) gmax[i] = 0ull;
    }
}
// sort each BS_CHUNK-sized chunk completely (k = 2 .. BS_CHUNK); direction alternates per chunk as bitonic needs
__global__ void __launch_bounds__(BS_THREADS) fs_sort_chunks_kernel(u64* __restrict__ keys) {
    __shared__ u64 s[BS_CHUNK];
    const int64_t base = (int64_t)blockIdx.x * BS_CHUNK;
    for (int i = threadIdx.x; i < BS_CHUNK; i += BS_THREADS) s[i] = keys[base + i];
    __syncthreads();
    for (int k = 2; k <= BS_CHUNK; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < BS_CHUNK; i += BS_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const int64_t gi = base + i;
                    const bool desc = ((gi & k) == 0);
                    const u64 a = s[i], b = s[ixj];
                    if (desc ? (a < b) : (a > b)) { s[i] = b; s[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < BS_CHUNK; i += BS_THREADS) keys[base + i] = s[i];
}
// one global compare-exchange step (j >= BS_CHUNK)
__global__ void fs_global_step_kernel(u64* __restrict__ keys, int64_t np2, int64_t j, int64_t k) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < (np2 >> 1); t += stride) {
        // t enumerates the pairs: insert a zero bit at position log2(j)
        const int64_t i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const int64_t ixj = i | j;
        const u64 a = keys[i], b = keys[ixj];
        const bool desc = ((i & k) == 0);
        if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[ixj] = a; }
    }
}
// the remaining steps j = BS_CHUNK/2 .. 1 of merge level k, fused in shared memory
__global__ void __launch_bounds__(BS_THREADS) fs_merge_chunks_kernel(u64* __restrict__ keys, int64_t k) {
    __shared__ u64 s[BS_CHUNK];
    const int64_t base = (int64_t)blockIdx.x * BS_CHUNK;
    for (int i = threadIdx.x; i < BS_CHUNK; i += BS_THREADS) s[i] = keys[base + i];
    __syncthreads();
    const bool desc = ((base & k) == 0);
    for (int j = BS_CHUNK >> 1; j > 0; j >>= 1) {
        for (int i = threadIdx.x; i < BS_CHUNK; i += BS_THREADS) {
            const int ixj = i ^ j;
            if (ixj > i) {
                const u64 a = s[i], b = s[ixj];
                if (desc ? (a < b) : (a > b)) { s[i] = b; s[ixj] = a; }
            }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < BS_CHUNK; i += BS_THREADS) keys[base + i] = s[i];
}
__global__ void fs_emit_kernel(const u64* __restrict__ keys, int64_t kk, const int64_t* __restrict__ ids, int64_t row0,
                               u64* __restrict__ out_keys, float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                               int32_t* __restrict__ out_count) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < kk; i += stride) {
        const u64 key = keys[i];
        const uint32_t row = key_row(key);
        const int64_t grow = row0 + (int64_t)row;
        out_keys[i] = (key & 0xffffffff00000000ull) | (u64)(uint32_t)(~(uint32_t)grow);
        out_scores[i] = key_score(key);
        out_ids[i] = ids ? ids[row] : grow;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *out_count = (int32_t)kk;
}

// Sort keys[0..np2) descending; np2 a power of two >= BS_CHUNK (pad with 0 = sorts last).
cudaError_t launch_sort_keys_desc(cudaStream_t st, u64* keys, int64_t np2)
{
    if (np2 < BS_CHUNK || (np2 & (np2 - 1))) return cudaErrorInvalidValue;
    const unsigned gblocks = (unsigned)((np2 / 256 < 4096) ? (np2 / 256) : 4096);
    const unsigned chunks = (unsigned)(np2 / BS_CHUNK);
    fs_sort_chunks_kernel<<<chunks, BS_THREADS, 0, st>>>(keys);
    int launches = 1;
    for (int64_t kl = (int64_t)BS_CHUNK << 1; kl <= np2; kl <<= 1) {
        for (int64_t j = kl >> 1; j >= BS_CHUNK; j >>= 1) {
            fs_global_step_kernel<<<gblocks, 256, 0, st>>>(keys, np2, j, kl);
            ++launches;
        }
        fs_merge_chunks_kernel<<<chunks, BS_THREADS, 0, st>>>(keys, kl);
        ++launches;
    }
    count_launch(launches);
    return cudaGetLastError();
}

cudaError_t launch_fullsort_topk(cudaStream_t st, const float* scores, int64_t n, u64* gmax, int group_shift,
                                 int64_t k, const int64_t* ids, int64_t row0, u64* sortbuf,
                                 u64* out_keys, float* out_scores, int64_t* out_ids, int32_t* out_count)
{
    if (n < 1 || k < 1) return cudaErrorInvalidValue;
    const int64_t kk = k < n ? k : n;
    int64_t np2 = next_pow2(n);
    if (np2 < BS_CHUNK) np2 = BS_CHUNK;
    const int64_t G = (n + ((int64_t)1 << group_shift) - 1) >> group_shift;
    const unsigned gblocks = (unsigned)((np2 / 256 < 4096) ? (np2 / 256) : 4096);
    fs_make_keys_kernel<<<gblocks, 256, 0, st>>>(scores, n, np2, sortbuf, gmax, G);
    cudaError_t se = launch_sort_keys_desc(st, sortbuf, np2);
    if (se != cudaSuccess) return se;
    count_launch(1);
    const unsigned eblocks = (unsigned)((kk + 255) / 256 < 1024 ? (kk + 255) / 256 : 1024);
    fs_emit_kernel<<<eblocks, 256, 0, st>>>(sortbuf, kk, ids, row0, out_keys, out_scores, out_ids, out_count);
    count_launch(1);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// cross-shard merge: n_lists candidate lists per query -> global top-k.  One CTA per query of the batch.
//
// Layout (all strides in ELEMENTS of the respective array): list l of query b has its keys at
// keys[l*list_stride + b*batch_stride + 0..cap), its ids at ids[same], and its valid count at
// counts[l*count_list_stride + b*count_batch_stride].  Outputs: out_*[b*k + 0..k), out_count[b].
// This covers both callers: the in-process engine (separate arrays, batch = 1) and the NCCL path
// (one packed int64 record [keys(k) | ids(k) | count] per query per rank, all-gathered).
// ---------------------------------------------------------------------------------------------
struct MergeLayout {
    int n_lists, cap, k;
    int64_t list_stride, batch_stride, count_list_stride, count_batch_stride;
    // verify_k >= 0 (batched records of the global-threshold path, batch.cu REFINE_PARTIAL | REFINE_DEFER): a list's count
    // word is the pair [count, ver]; count < 0 on any list, or sum(ver) < verify_k, means the coarse pass could not vouch
    // for this query: out_count = -1 and the caller redoes it with the exact kernels.  Lists may be TRUNCATED (bit 30 of
    // count: the rank had more entries than the record holds, cap < k): fine as long as the list's last shipped entry
    // does not make the global top k -- then nothing behind it can; otherwise -1 as well.
    int verify_k;
    const int* abort_flag;       // optional device word: non-zero = the records never arrived (peer exchange timed out)
};
constexpr int32_t RECORD_TRUNCATED = 1 << 30;

// true: the query's records are good.  All threads call it; uses sm.bcast32[0..2] ([2] = bit l set: list l is truncated,
// l < 31 -- the launcher keeps n_lists <= 16 when records may be truncated).
__device__ inline bool merge_records_verified(SelectSmem& sm, const int32_t* counts, const MergeLayout& L) {
    const int tid = threadIdx.x;
    if (tid == 0) { sm.bcast32[0] = 0; sm.bcast32[1] = 0; sm.bcast32[2] = 0; }
    __syncthreads();
    if (tid < L.n_lists) {
        const int32_t* c = counts + (int64_t)tid * L.count_list_stride;
        if (c[0] < 0) atomicOr(&sm.bcast32[0], 1);
        else atomicAdd(&sm.bcast32[1], max(0, c[1]));
        if (c[0] >= 0 && (c[0] & RECORD_TRUNCATED)) atomicOr(&sm.bcast32[2], 1 << min(tid, 30));
    }
    __syncthreads();
    const bool ok = sm.bcast32[0] == 0 && sm.bcast32[1] >= L.verify_k;
    __syncthreads();
    return ok;
}

// Rank merge of n_lists lists that are each sorted descending (what the selection / refine kernels emit): list l sits at
// sm.sortbuf[off[l] .. off[l] + cnt[l]) with its payload beside it; keys are unique (the row is in the low word), so the
// global rank of an element is its index in its own list plus, for every other list, the number of keys greater than
// it (one binary search each).  Elements of rank < kk go straight to the output: no sort, no second buffer.
// Returns false (nothing written) if some list is not sorted; the caller then takes the bitonic path.
// trunc_mask / k_full / trunc_bad (optional): bit l of trunc_mask = list l was truncated by its sender; *trunc_bad is set
// when such a list's last entry has rank < k_full, i.e. entries the sender did not ship could belong to the top k_full.
__device__ bool rank_merge_emit(SelectSmem& sm, int n_lists, const uint32_t* cnt, const uint32_t* off, int total, int kk,
                                float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                                uint32_t trunc_mask = 0, int k_full = 0, int* trunc_bad = nullptr)
{
    const int tid = threadIdx.x;
    __shared__ int unsorted;
    if (tid == 0) unsorted = 0;
    __syncthreads();
    for (int i = tid; i < total; i += blockDim.x) {
        int l = 0;
        while (l + 1 < n_lists && (uint32_t)i >= off[l + 1]) ++l;
        if ((uint32_t)i > off[l] && sm.sortbuf[i] >= sm.sortbuf[i - 1]) unsorted = 1;
    }
    __syncthreads();
    if (unsorted) return false;
    for (int i = tid; i < total; i += blockDim.x) {
        int l = 0;
        while (l + 1 < n_lists && (uint32_t)i >= off[l + 1]) ++l;
        const u64 key = sm.sortbuf[i];
        int rank = i - (int)off[l];
        for (int m = 0; m < n_lists; ++m) {
            if (m == l) continue;
            int lo = (int)off[m], hi = lo + (int)cnt[m];               // first position in list m whose key is < mine
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (sm.sortbuf[mid] > key) lo = mid + 1; else hi = mid; }
            rank += lo - (int)off[m];
        }
        if (rank < kk) { out_scores[rank] = key_score(key); out_ids[rank] = sm.payload[i]; }
        if (trunc_mask && ((trunc_mask >> l) & 1u) && i == (int)(off[l] + cnt[l]) - 1 && rank < k_full) *trunc_bad = 1;
    }
    return true;
}

__global__ void __launch_bounds__(SEL_THREADS, 1)
merge_lists_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ ids, const int32_t* __restrict__ counts,
                   MergeLayout L, float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                   int32_t* __restrict__ out_count)
{
    extern __shared__ __align__(16) unsigned char sel_smem_raw[];
    SelectSmem& sm = *reinterpret_cast<SelectSmem*>(sel_smem_raw);
    const int tid = threadIdx.x, b = blockIdx.x;
    keys += (int64_t)b * L.batch_stride; ids += (int64_t)b * L.batch_stride;
    counts += (int64_t)b * L.count_batch_stride;
    out_scores += (int64_t)b * L.k; out_ids += (int64_t)b * L.k;
    uint32_t* cnt = sm.hist;                                  // per-list counts and offsets (list order is kept);
    uint32_t* off = sm.hist + 1024;                           // n_lists <= 1023 (launcher)
    if (L.abort_flag && *L.abort_flag) { if (tid == 0) out_count[b] = MERGE_WINDOW_TIMED_OUT; return; }
    if (L.verify_k >= 0 && !merge_records_verified(sm, counts, L)) { if (tid == 0) out_count[b] = -1; return; }
    const uint32_t trunc_mask = L.verify_k >= 0 ? (uint32_t)sm.bcast32[2] : 0u;
    __shared__ int trunc_bad;
    if (tid == 0) trunc_bad = 0;
    if (tid < L.n_lists) {
        int32_t c = counts[(int64_t)tid * L.count_list_stride];
        if (L.verify_k >= 0) c &= ~RECORD_TRUNCATED;
        cnt[tid] = (uint32_t)max(0, min(c, L.cap));
    }
    __syncthreads();
    if (tid == 0) { uint32_t o = 0; for (int l = 0; l < L.n_lists; ++l) { off[l] = o; o += cnt[l]; } off[L.n_lists] = o; }
    __syncthreads();
    const int span = L.n_lists * L.cap;                       // <= SORT_CAP (host guarantees)
    for (int i = tid; i < span; i += blockDim.x) {
        const int l = i / L.cap, p = i - l * L.cap;
        if ((uint32_t)p < cnt[l]) {
            sm.sortbuf[off[l] + p] = keys[(int64_t)l * L.list_stride + p];
            sm.payload[off[l] + p] = ids[(int64_t)l * L.list_stride + p];
        }
    }
    __syncthreads();
    const int total = (int)off[L.n_lists];
    const int kk = min(L.k, total);
    if (rank_merge_emit(sm, L.n_lists, cnt, off, total, kk, out_scores, out_ids, trunc_mask, L.k, &trunc_bad)) {
        __syncthreads();
        if (tid == 0) out_count[b] = trunc_bad ? -1 : kk;
        return;
    }
    if (L.verify_k >= 0) { if (tid == 0) out_count[b] = -1; return; }     // verified records are always sorted
    int np2 = 1; while (np2 < total) np2 <<= 1;
    for (int i = total + tid; i < np2; i += blockDim.x) { sm.sortbuf[i] = 0ull; sm.payload[i] = -1; }
    __syncthreads();
    block_bitonic_desc<true>(sm.sortbuf, sm.payload, np2);
    for (int i = tid; i < kk; i += blockDim.x) { out_scores[i] = key_score(sm.sortbuf[i]); out_ids[i] = sm.payload[i]; }
    if (tid == 0) out_count[b] = kk;
}

// The same merge for SMALL records (n_lists <= 32, n_lists * cap <= 1024: batched records of 2..16 ranks): 256 threads and
// 17 KB of shared memory, so eight CTAs share an SM instead of two -- a 1024-query batch is one wave, not four.
constexpr int MERGE_SMALL_THREADS = 256;
constexpr int MERGE_SMALL_SPAN = 1024;
__global__ void __launch_bounds__(MERGE_SMALL_THREADS)
merge_lists_small_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ ids, const int32_t* __restrict__ counts,
                         MergeLayout L, float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                         int32_t* __restrict__ out_count)
{
    __shared__ u64 sk[MERGE_SMALL_SPAN];
    __shared__ int64_t sp[MERGE_SMALL_SPAN];
    __shared__ uint32_t cnt[32], off[33];
    __shared__ int s_bad, s_ver, s_unsorted;
    __shared__ uint32_t s_trunc;
    const int tid = threadIdx.x, b = blockIdx.x;
    keys += (int64_t)b * L.batch_stride; ids += (int64_t)b * L.batch_stride;
    counts += (int64_t)b * L.count_batch_stride;
    out_scores += (int64_t)b * L.k; out_ids += (int64_t)b * L.k;
    if (L.abort_flag && *L.abort_flag) { if (tid == 0) out_count[b] = MERGE_WINDOW_TIMED_OUT; return; }
    if (tid == 0) { s_bad = 0; s_ver = 0; s_unsorted = 0; s_trunc = 0; }
    __syncthreads();
    if (tid < L.n_lists) {
        const int32_t* cw = counts + (int64_t)tid * L.count_list_stride;
        int32_t c = cw[0];
        if (L.verify_k >= 0) {
            if (c < 0) atomicOr(&s_bad, 1);
            else { atomicAdd(&s_ver, max(0, cw[1])); if (c & RECORD_TRUNCATED) atomicOr(&s_trunc, 1u << tid); }
            c &= ~RECORD_TRUNCATED;
        }
        cnt[tid] = (uint32_t)max(0, min(c, L.cap));
    }
    __syncthreads();
    if (L.verify_k >= 0 && (s_bad || s_ver < L.verify_k)) { if (tid == 0) out_count[b] = -1; return; }
    if (tid == 0) { uint32_t o = 0; for (int l = 0; l < L.n_lists; ++l) { off[l] = o; o += cnt[l]; } off[L.n_lists] = o; }
    __syncthreads();
    const int span = L.n_lists * L.cap;
    for (int i = tid; i < span; i += MERGE_SMALL_THREADS) {
        const int l = i / L.cap, p = i - l * L.cap;
        if ((uint32_t)p < cnt[l]) {
            sk[off[l] + p] = keys[(int64_t)l * L.list_stride + p];
            sp[off[l] + p] = ids[(int64_t)l * L.list_stride + p];
        }
    }
    __syncthreads();
    const int total = (int)off[L.n_lists];
    const int kk = min(L.k, total);
    const uint32_t trunc = s_trunc;
    for (int i = tid; i < total; i += MERGE_SMALL_THREADS) {
        int l = 0;
        while (l + 1 < L.n_lists && (uint32_t)i >= off[l + 1]) ++l;
        if ((uint32_t)i > off[l] && sk[i] >= sk[i - 1]) s_unsorted = 1;
    }
    __syncthreads();
    const bool sorted = s_unsorted == 0;
    __syncthreads();
    for (int i = tid; i < total; i += MERGE_SMALL_THREADS) {
        int l = 0;
        while (l + 1 < L.n_lists && (uint32_t)i >= off[l + 1]) ++l;
        const u64 key = sk[i];
        int rank = 0;
        if (sorted) {                                         // position in its own list + binary searches in the others
            rank = i - (int)off[l];
            for (int m = 0; m < L.n_lists; ++m) {
                if (m == l) continue;
                int lo = (int)off[m], hi = lo + (int)cnt[m];
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (sk[mid] > key) lo = mid + 1; else hi = mid; }
                rank += lo - (int)off[m];
            }
        } else {                                              // a list out of order (stateless callers only): count
            for (int j = 0; j < total; ++j) rank += sk[j] > key ? 1 : 0;
        }
        if (rank < kk) { out_scores[rank] = key_score(key); out_ids[rank] = sp[i]; }
        if (((trunc >> l) & 1u) && i == (int)(off[l] + cnt[l]) - 1 && rank < L.k) s_bad = 1;
    }
    __syncthreads();
    if (tid == 0) out_count[b] = s_bad ? -1 : kk;
}

// Generic merge for n_lists * cap > SORT_CAP: compact valid entries into scratch, select, sort.
__global__ void __launch_bounds__(SEL_THREADS, 1)
merge_lists_big_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ ids, const int32_t* __restrict__ counts,
                       MergeLayout L, u64* sk, int64_t* sp, float* __restrict__ out_scores,
                       int64_t* __restrict__ out_ids, int32_t* __restrict__ out_count)
{
    extern __shared__ __align__(16) unsigned char sel_smem_raw[];
    SelectSmem& sm = *reinterpret_cast<SelectSmem*>(sel_smem_raw);
    const int tid = threadIdx.x, b = blockIdx.x;
    const int64_t span = (int64_t)L.n_lists * L.cap;
    keys += (int64_t)b * L.batch_stride; ids += (int64_t)b * L.batch_stride;
    counts += (int64_t)b * L.count_batch_stride;
    out_scores += (int64_t)b * L.k; out_ids += (int64_t)b * L.k;
    sk += (int64_t)b * span; sp += (int64_t)b * span;
    if (L.abort_flag && *L.abort_flag) { if (tid == 0) out_count[b] = MERGE_WINDOW_TIMED_OUT; return; }
    if (L.verify_k >= 0 && (!merge_records_verified(sm, counts, L) || sm.bcast32[2] != 0)) { if (tid == 0) out_count[b] = -1; return; }
    if (tid == 0) sm.counter = 0;
    __syncthreads();
    for (int64_t i = tid; i < span; i += blockDim.x) {
        const int l = (int)(i / L.cap), p = (int)(i - (int64_t)l * L.cap);
        if (p < min(counts[(int64_t)l * L.count_list_stride] & (L.verify_k >= 0 ? ~RECORD_TRUNCATED : -1), L.cap)) {
            const uint32_t slot = atomicAdd(&sm.counter, 1u);
            sk[slot] = keys[(int64_t)l * L.list_stride + p];
            sp[slot] = ids[(int64_t)l * L.list_stride + p];
        }
    }
    __syncthreads();
    const int total = (int)sm.counter;
    const int kk = min(L.k, total);
    __syncthreads();
    if (kk == 0) { if (tid == 0) out_count[b] = 0; return; }
    u64 tau = 0;
    if (total > kk) tau = block_kth_largest(sk, total, kk, sm);
    if (tid == 0) sm.counter = 0;
    __syncthreads();
    for (int i = tid; i < total; i += blockDim.x) {
        const u64 v = sk[i];
        if (v >= tau) { const uint32_t slot = atomicAdd(&sm.counter, 1u); if (slot < (uint32_t)SORT_CAP) { sm.sortbuf[slot] = v; sm.payload[slot] = sp[i]; } }
    }
    __syncthreads();
    const int c = (int)min(sm.counter, (uint32_t)SORT_CAP);
    int np2 = 1; while (np2 < c) np2 <<= 1;
    for (int i = c + tid; i < np2; i += blockDim.x) { sm.sortbuf[i] = 0ull; sm.payload[i] = -1; }
    __syncthreads();
    block_bitonic_desc<true>(sm.sortbuf, sm.payload, np2);
    for (int i = tid; i < kk; i += blockDim.x) { out_scores[i] = key_score(sm.sortbuf[i]); out_ids[i] = sm.payload[i]; }
    if (tid == 0) out_count[b] = kk;
}

cudaError_t launch_merge_ex(cudaStream_t st, const u64* keys, const int64_t* ids, const int32_t* counts,
                            int n_lists, int cap, int k, int batch, int64_t list_stride, int64_t batch_stride,
                            int64_t count_list_stride, int64_t count_batch_stride,
                            u64* scratch_keys, int64_t* scratch_ids,
                            float* out_scores, int64_t* out_ids, int32_t* out_count, int verify_k, const int* abort_flag)
{
    if (n_lists < 1 || n_lists > 1023 || cap < 1 || k < 1 || k > K_FAST_MAX || batch < 1) return cudaErrorInvalidValue;
    static bool attr_set[64][2] = {{false}};
    int dev = 0; cudaGetDevice(&dev);
    const bool big = (int64_t)n_lists * cap > SORT_CAP;
    if (dev >= 0 && dev < 64 && !attr_set[dev][big]) {
        cudaError_t e = big
            ? cudaFuncSetAttribute(merge_lists_big_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectSmem))
            : cudaFuncSetAttribute(merge_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectSmem));
        if (e != cudaSuccess) return e;
        attr_set[dev][big] = true;
    }
    MergeLayout L{n_lists, cap, k, list_stride, batch_stride, count_list_stride, count_batch_stride, verify_k, abort_flag};
    static const bool small_off = [] { const char* v = getenv("SVSB_MERGE_SMALL"); return v && atoi(v) == 0; }();
    if (!small_off && batch >= 8 && n_lists <= 32 && (int64_t)n_lists * cap <= MERGE_SMALL_SPAN) {
        merge_lists_small_kernel<<<batch, MERGE_SMALL_THREADS, 0, st>>>(keys, ids, counts, L, out_scores, out_ids, out_count);
        count_launch();
        return cudaGetLastError();
    }
    if (big) {
        if (!scratch_keys || !scratch_ids) return cudaErrorInvalidValue;
        merge_lists_big_kernel<<<batch, SEL_THREADS, sizeof(SelectSmem), st>>>(keys, ids, counts, L, scratch_keys, scratch_ids,
                                                                              out_scores, out_ids, out_count);
    } else {
        merge_lists_kernel<<<batch, SEL_THREADS, sizeof(SelectSmem), st>>>(keys, ids, counts, L, out_scores, out_ids, out_count);
    }
    count_launch();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Merge of a gather-window slot (peer exchange): the lists were stored by the other ranks' selection kernels over
// peer memory.  Thread r waits for rank r's flag (acquire, system scope), then the CTA merges exactly like
// merge_lists_kernel / merge_lists_big_kernel -- with L1-bypassing loads, since this SM may hold stale lines of
// the slot from its previous use.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SEL_THREADS, 1)
merge_window_kernel(const u64* slot_base, const u64* flags, u64 seq, int world, int cap, int k, u64 timeout_ns,
                    u64* sk, int64_t* sp, float* __restrict__ out_scores, int64_t* __restrict__ out_ids,
                    int32_t* __restrict__ out_count, u64* __restrict__ stamps)
{
    extern __shared__ __align__(16) unsigned char sel_smem_raw[];
    SelectSmem& sm = *reinterpret_cast<SelectSmem*>(sel_smem_raw);
    const int tid = threadIdx.x;
    const int64_t rec_words = 2 * (int64_t)cap + 2;
    pdl_wait();                                    // scratch / outputs may still be in use by the previous kernel
    if (tid == 0) sm.counter = 0;
    // measurement aid (SVSB_XCHG_STAMPS=1): when did this merge start, when had rank r's record arrived (%globaltimer, ns)
    if (stamps && tid == 0) { u64 t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); stamps[0] = seq; stamps[1] = t_; }
    __syncthreads();
    if (tid < world) {
        // A peer that died or left the SPMD sequence must not hang this GPU: give up after timeout_ns and report it.
        unsigned ns = 32;
        u64 t0 = 0;
        while (ld_acquire_sys(flags + tid) < seq) {
            __nanosleep(ns);
            if (ns < 1024) ns <<= 1;
            else {
                u64 now; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (t0 == 0) t0 = now;
                else if (now - t0 > timeout_ns) { atomicAdd(&sm.counter, 1u); break; }
            }
        }
        if (stamps) { u64 t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); stamps[4 + tid] = t_; }
    }
    __syncthreads();
    if (sm.counter != 0) { if (tid == 0) *out_count = MERGE_WINDOW_TIMED_OUT; return; }
    __syncthreads();
    const bool big = sk != nullptr;                            // world * k > SORT_CAP: compact into global scratch
    const int span = world * k;
    if (!big) {
        // lists kept in order in shared memory, then the rank merge (each rank's record is sorted descending)
        uint32_t* cnt = sm.hist;
        uint32_t* off = sm.hist + 64;
        if (tid < world) cnt[tid] = (uint32_t)min((u64)k, __ldcg(slot_base + (int64_t)tid * rec_words + 2 * cap));
        __syncthreads();
        if (tid == 0) { uint32_t o = 0; for (int l = 0; l < world; ++l) { off[l] = o; o += cnt[l]; } off[world] = o; }
        __syncthreads();
        for (int i = tid; i < span; i += blockDim.x) {
            const int l = i / k, p = i - l * k;
            const u64* rec = slot_base + (int64_t)l * rec_words;
            if ((uint32_t)p < cnt[l]) {
                sm.sortbuf[off[l] + p] = __ldcg(rec + p);
                sm.payload[off[l] + p] = (int64_t)__ldcg(rec + cap + p);
            }
        }
        __syncthreads();
        const int total_s = (int)off[world];
        const int kk_s = min(k, total_s);
        if (rank_merge_emit(sm, world, cnt, off, total_s, kk_s, out_scores, out_ids)) {
            if (tid == 0) *out_count = kk_s;
            if (stamps && tid == 0) { u64 t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); stamps[2] = t_; }
            return;
        }
        if (tid == 0) sm.counter = (uint32_t)total_s;         // unsorted input: fall through to the bitonic sort
        __syncthreads();
    } else {
        for (int i = tid; i < span; i += blockDim.x) {
            const int l = i / k, p = i - l * k;
            const u64* rec = slot_base + (int64_t)l * rec_words;
            if (p < (int)min((u64)k, __ldcg(rec + 2 * cap))) {
                const uint32_t slot = atomicAdd(&sm.counter, 1u);
                sk[slot] = __ldcg(rec + p); sp[slot] = (int64_t)__ldcg(rec + cap + p);
            }
        }
        __syncthreads();
    }
    const int total = (int)sm.counter;
    const int kk = min(k, total);
    __syncthreads();
    if (kk == 0) { if (tid == 0) *out_count = 0; return; }
    int c = total;
    if (big) {
        u64 tau = 0;
        if (total > kk) tau = block_kth_largest(sk, total, kk, sm);
        if (tid == 0) sm.counter = 0;
        __syncthreads();
        for (int i = tid; i < total; i += blockDim.x) {
            const u64 v = sk[i];
            if (v >= tau) { const uint32_t slot = atomicAdd(&sm.counter, 1u); if (slot < (uint32_t)SORT_CAP) { sm.sortbuf[slot] = v; sm.payload[slot] = sp[i]; } }
        }
        __syncthreads();
        c = (int)min(sm.counter, (uint32_t)SORT_CAP);
    }
    int np2 = 1; while (np2 < c) np2 <<= 1;
    for (int i = c + tid; i < np2; i += blockDim.x) { sm.sortbuf[i] = 0ull; sm.payload[i] = -1; }
    __syncthreads();
    block_bitonic_desc<true>(sm.sortbuf, sm.payload, np2);
    for (int i = tid; i < kk; i += blockDim.x) { out_scores[i] = key_score(sm.sortbuf[i]); out_ids[i] = sm.payload[i]; }
    if (tid == 0) *out_count = kk;
}

// ---------------------------------------------------------------------------------------------
// Large-k merge (k > K_FAST_MAX across several devices, e.g. the notebooks' n = len(kb) full ranking on a row-sharded
// matrix): every list is sorted descending and keys are unique, so an element's global rank is its index in its own
// list plus, per other list, the number of greater keys (one binary search each, lists are L2-resident).  Elements of
// rank < k go straight to the output; no sort, any k.
// List l holds at most cap entries at keys / ids [l * list_stride ..); its count is counts[l * count_stride].  A count
// outside [0, cap] (negative, or RECORD_TRUNCATED set: the list lost entries) makes the whole merge unanswerable: the
// kernel writes nothing but out_count = -1, since a missing entry could belong anywhere in the top k.
// ---------------------------------------------------------------------------------------------
__global__ void merge_sorted_big_kernel(const u64* __restrict__ keys, const int64_t* __restrict__ ids, const int32_t* __restrict__ counts,
                                        int n_lists, int64_t cap, int64_t list_stride, int64_t count_stride, int64_t k,
                                        float* __restrict__ out_scores, int64_t* __restrict__ out_ids, int32_t* __restrict__ out_count)
{
    int64_t total = 0;
    for (int l = 0; l < n_lists; ++l) {
        const int32_t c = counts[l * count_stride];
        if (c < 0 || c > cap) {
            if (blockIdx.x == 0 && threadIdx.x == 0) *out_count = -1;
            return;
        }
        total += c;
    }
    const int64_t kk = k < total ? k : total;
    const int64_t span = (int64_t)n_lists * cap;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < span; e += step) {
        const int l = (int)(e / cap);
        const int64_t p = e - (int64_t)l * cap;
        if (p >= counts[l * count_stride]) continue;
        const int64_t at = (int64_t)l * list_stride + p;
        const u64 key = keys[at];
        int64_t rank = p;
        for (int m = 0; m < n_lists && rank < kk; ++m) {
            if (m == l) continue;
            const u64* lm = keys + (int64_t)m * list_stride;
            int64_t lo = 0, hi = counts[m * count_stride];                          // first position whose key is < mine
            while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (lm[mid] > key) lo = mid + 1; else hi = mid; }
            rank += lo;
        }
        if (rank < kk) { out_scores[rank] = key_score(key); out_ids[rank] = ids[at]; }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *out_count = (int32_t)kk;
}

cudaError_t launch_merge_sorted_big(cudaStream_t st, const u64* keys, const int64_t* ids, const int32_t* counts, int n_lists,
                                    int64_t cap, int64_t list_stride, int64_t count_stride, int64_t k, float* out_scores,
                                    int64_t* out_ids, int32_t* out_count)
{
    if (n_lists < 1 || cap < 1 || list_stride < cap || count_stride < 1 || k < 1) return cudaErrorInvalidValue;
    const int64_t span = (int64_t)n_lists * cap;
    const unsigned blocks = (unsigned)std::min<int64_t>((span + 255) / 256, 148 * 8);
    merge_sorted_big_kernel<<<blocks, 256, 0, st>>>(keys, ids, counts, n_lists, cap, list_stride, count_stride, k, out_scores,
                                                    out_ids, out_count);
    count_launch();
    return cudaGetLastError();
}

// The same rank merge for the per-device lists of the pairwise pass (multi.cu): an entry is (score, row a, row b) and
// orders by (ordered score desc, then the 64-bit pair a << 32 | b asc) -- a 96-bit key, unique because every pair of
// rows is scored on exactly one device.  The rows of the top k are mapped to embeddings.ids on the way out.
__device__ __forceinline__ bool pair_before(uint32_t so, u64 sp, uint32_t to, u64 tp) { return so > to || (so == to && sp < tp); }

__global__ void merge_sorted_pairs_kernel(const float* __restrict__ scores, const int64_t* __restrict__ rows_a,
                                          const int64_t* __restrict__ rows_b, const int32_t* __restrict__ counts, int n_lists,
                                          int64_t stride, int64_t k, const __grid_constant__ PairRows rows,
                                          float* __restrict__ out_scores, int64_t* __restrict__ out_a, int64_t* __restrict__ out_b,
                                          int32_t* __restrict__ out_count)
{
    int64_t total = 0;
    for (int l = 0; l < n_lists; ++l) total += min((int64_t)max(counts[l], 0), stride);
    const int64_t kk = k < total ? k : total;
    const int64_t span = (int64_t)n_lists * stride;
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < span; e += step) {
        const int l = (int)(e / stride);
        const int64_t p = e - (int64_t)l * stride;
        if (p >= min((int64_t)max(counts[l], 0), stride)) continue;
        const float sc = scores[e];
        const uint32_t so = f32_to_ordered(sc);
        const u64 sp = ((u64)rows_a[e] << 32) | (u64)rows_b[e];
        int64_t rank = p;
        for (int m = 0; m < n_lists && rank < kk; ++m) {
            if (m == l) continue;
            const int64_t base = (int64_t)m * stride;
            int64_t lo = 0, hi = min((int64_t)max(counts[m], 0), stride);          // first entry of list m not before mine
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                const u64 tp = ((u64)rows_a[base + mid] << 32) | (u64)rows_b[base + mid];
                if (pair_before(f32_to_ordered(scores[base + mid]), tp, so, sp)) lo = mid + 1; else hi = mid;
            }
            rank += lo;
        }
        if (rank < kk) {
            const int64_t a = rows_a[e], b = rows_b[e];
            const int s_a = rows.shard_of(a), s_b = rows.shard_of(b);
            out_scores[rank] = sc;
            out_a[rank] = rows.ids[s_a][a - rows.row0[s_a]];
            out_b[rank] = rows.ids[s_b][b - rows.row0[s_b]];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *out_count = (int32_t)kk;
}

cudaError_t launch_merge_sorted_pairs(cudaStream_t st, const float* scores, const int64_t* rows_a, const int64_t* rows_b,
                                      const int32_t* counts, int n_lists, int64_t stride, int64_t k, const PairRows& rows,
                                      float* out_scores, int64_t* out_a, int64_t* out_b, int32_t* out_count)
{
    if (n_lists < 1 || n_lists > XCHG_MAX_RANKS || stride < 1 || k < 1) return cudaErrorInvalidValue;
    const int64_t span = (int64_t)n_lists * stride;
    const unsigned blocks = (unsigned)std::min<int64_t>((span + 255) / 256, 148 * 8);
    merge_sorted_pairs_kernel<<<blocks, 256, 0, st>>>(scores, rows_a, rows_b, counts, n_lists, stride, k, rows, out_scores, out_a, out_b, out_count);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_merge_window(cudaStream_t st, const u64* slot_base, const u64* flags, unsigned long long seq,
                                int world, int cap, int k, unsigned long long timeout_ns, u64* scratch_keys, int64_t* scratch_ids,
                                float* out_scores, int64_t* out_ids, int32_t* out_count, u64* stamps)
{
    if (world < 1 || world > XCHG_MAX_RANKS || k < 1 || k > K_FAST_MAX || cap < k) return cudaErrorInvalidValue;
    static bool attr_set[64] = {false};
    int dev = 0; cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && !attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(merge_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectSmem));
        if (e != cudaSuccess) return e;
        attr_set[dev] = true;
    }
    const bool big = (int64_t)world * k > SORT_CAP;
    if (big && (!scratch_keys || !scratch_ids)) return cudaErrorInvalidValue;
    cudaError_t le = launch_kernel(merge_window_kernel, dim3(1), dim3(SEL_THREADS), sizeof(SelectSmem), st, slot_base, flags, (u64)seq, world, cap, k,
                                   (u64)timeout_ns, big ? scratch_keys : (u64*)nullptr, big ? scratch_ids : (int64_t*)nullptr,
                                   out_scores, out_ids, out_count, stamps);
    count_launch();
    return le != cudaSuccess ? le : cudaGetLastError();
}

cudaError_t preload_peer_kernels()
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, select_topk_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, merge_window_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, push_empty_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, stage_query_kernel);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(select_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectKeysSmem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(merge_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SelectSmem));
    return e;
}

cudaError_t preload_merge_kernels()
{
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, merge_lists_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, merge_lists_big_kernel);
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, merge_lists_small_kernel);
    return e;
}

cudaError_t launch_merge(cudaStream_t st, const u64* keys, const int64_t* ids, const int32_t* counts,
                         int n_lists, int stride, int k, u64* scratch_keys, int64_t* scratch_ids,
                         float* out_scores, int64_t* out_ids, int32_t* out_count)
{
    return launch_merge_ex(st, keys, ids, counts, n_lists, stride, k, 1, stride, 0, 1, 0,
                           scratch_keys, scratch_ids, out_scores, out_ids, out_count);
}

}  // namespace svsb
