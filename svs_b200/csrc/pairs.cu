// Pairwise top pairs on the batched contraction (SURVEY.md section 8f rank 2).
//
// Replaces the compute of document_top_pairwise_scores (reference src/svs/kb.py:1642-1671, 1208-1243):
// `np.dot(M, M.T)` -- an N x N fp32 SGEMM whose result the reference materialises (95 MB at 4,875 docs, impossible
// at 1M) -- followed by get_top_pairs (src/svs/util.py:206-233: upper triangle without the diagonal, argpartition,
// sort).  Here the N x N scores are never written: blocks of <= 2048 rows play the "queries" of the coarse tensor
// core pass (coarse.cu, pairwise mode: only row > query row counts, tiles under the diagonal are skipped), ONE global
// threshold filters them, and the survivors are re-scored exactly in fp32.  The threshold tightens block after
// block: it is (the n-th largest coarse score among the pairs seen so far) - 2 eps, a valid lower bound for
// (final n-th largest coarse) - 2 eps, so every pair that can be in the exact top-n stays in the list (same argument
// as batch.cu with the global list in place of a query's list).
// Multi-device engines (multi.cu: multi_top_pairs) run the same pass per device over a share of the pairs -- the
// triangle of the own shard plus rectangles against blocks of the peers' rows -- with one threshold per device; pairs
// are kept in global rows and the re-score reads rows through a table of shard pointers (PairRows, peer memory).
//
// Order of the result: score descending, then row index of the first document ascending, then of the second
// (the reference orders exact ties by descending flat index of the upper triangle, src/svs/util.py:203).
#include "select_common.cuh"

#include <cuda_fp16.h>

namespace svsb {

constexpr int PR_THREADS = 1024;
constexpr int PR_BINS = KTH_BINS;
constexpr int PR_SMALL = KTH_SMALL;

// thr[q] = *scalar for q < b, +inf for the padding queries
__global__ void pairs_fill_thr_kernel(float* __restrict__ thr, int b_pad, int b, const float* __restrict__ scalar) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < b_pad) thr[q] = q < b ? *scalar : __int_as_float(0x7f800000);
}

// Append the block's per-query candidate lists to the global pair list.  One CTA per query row.  Query q is global
// row q_row0 + q, matrix row r (the key's row) global row m_row0 + r; the pair goes in as (smaller row, larger row).
// state[0] = list count, state[1] = error flags (1: a per-query list overflowed, 2: the global list overflowed)
__global__ void __launch_bounds__(256)
pairs_gather_kernel(const u64* __restrict__ cand, const int32_t* __restrict__ cand_cnt, int cand_cap, int64_t q_row0, int64_t m_row0,
                    uint32_t* __restrict__ list_o, u64* __restrict__ list_pair, int64_t list_cap, unsigned long long* state)
{
    __shared__ unsigned long long base;
    const int q = blockIdx.x;
    const int cnt = cand_cnt[q];
    if (cnt <= 0) return;
    if (cnt > cand_cap) { if (threadIdx.x == 0) atomicOr(&state[1], 1ull); return; }
    if (threadIdx.x == 0) base = atomicAdd(&state[0], (unsigned long long)cnt);
    __syncthreads();
    const unsigned long long b0 = base;
    if (b0 + (unsigned long long)cnt > (unsigned long long)list_cap) { if (threadIdx.x == 0) atomicOr(&state[1], 2ull); return; }
    const u64* cq = cand + (size_t)q * cand_cap;
    const u64 i = (u64)(q_row0 + q);
    for (int c = threadIdx.x; c < cnt; c += blockDim.x) {
        const u64 key = cq[c];
        const u64 j = (u64)(m_row0 + (int64_t)key_row(key));
        list_o[b0 + c] = (uint32_t)(key >> 32);
        list_pair[b0 + c] = i < j ? (i << 32) | j : (j << 32) | i;
    }
}

// Single CTA: tighten the global threshold to (n-th largest coarse score in the list) - 2 eps.
// Also usable on the coarse kernel's fp16 sample dump (vals != nullptr): the bootstrap.
__global__ void __launch_bounds__(PR_THREADS)
pairs_tau_kernel(const uint32_t* __restrict__ list_o, const __half* __restrict__ vals, int64_t vals_count,
                 const unsigned long long* __restrict__ state, int64_t list_cap, int n, float eps2, float* __restrict__ thr_scalar)
{
    __shared__ uint32_t hist[PR_BINS];
    __shared__ uint32_t scratch[72];
    __shared__ uint32_t small[PR_SMALL];
    int64_t count = vals ? vals_count : (int64_t)min(state[0], (unsigned long long)list_cap);
    if (count < n) return;
    uint32_t o;
    if (vals) o = block_kth_largest_o32([&](int64_t i) { return f32_to_ordered(__half2float(vals[i])); }, count, n, hist, scratch, small);
    else      o = block_kth_largest_o32([&](int64_t i) { return list_o[i]; }, count, n, hist, scratch, small);
    if (threadIdx.x == 0) {
        const float t = ordered_to_f32(o) - eps2;
        if (t > *thr_scalar) *thr_scalar = t;            // -inf sample entries (masked pairs) give t = -inf: no change
    }
}

// dst = entries of src with coarse score >= threshold.  dst_state[0] must be zero on entry.
__global__ void __launch_bounds__(256)
pairs_compact_kernel(const uint32_t* __restrict__ src_o, const u64* __restrict__ src_pair, const unsigned long long* __restrict__ src_state,
                     int64_t list_cap, uint32_t* __restrict__ dst_o, u64* __restrict__ dst_pair, unsigned long long* dst_state,
                     const float* __restrict__ thr_scalar)
{
    const int64_t count = (int64_t)min(src_state[0], (unsigned long long)list_cap);
    const float thr = *thr_scalar;
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t rounds = (count + stride - 1) / stride;
    for (int64_t r = 0; r < rounds; ++r) {
        const int64_t i = r * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        bool keep = false; uint32_t o = 0; u64 pr = 0;
        if (i < count) { o = src_o[i]; pr = src_pair[i]; keep = ordered_to_f32(o) >= thr; }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (m) {
            unsigned long long b0 = 0;
            if (lane == 0) b0 = atomicAdd(&dst_state[0], (unsigned long long)__popc(m));
            b0 = __shfl_sync(0xffffffffu, b0, 0);
            if (keep) { const unsigned long long p = b0 + __popc(m & ((1u << lane) - 1u)); dst_o[p] = o; dst_pair[p] = pr; }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) dst_state[1] = src_state[1];     // carry the error flags
}

// keys[c] = ~pair for c < count (descending sort of ~pair == ascending (i, j)), 0 for the power-of-two padding
__global__ void pairs_sortkeys_kernel(const u64* __restrict__ list_pair, int64_t count, int64_t np2, u64* __restrict__ keys) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < np2; c += stride) keys[c] = c < count ? ~list_pair[c] : 0ull;
}

// exact fp32 score of pair c = (i, j) (keys sorted, ~pair; global rows, both rows found through the shard table), one
// warp per pair, the similarity kernel's summation order with row i in the role of the query.  fma(m, q, acc) ==
// fma(q, m, acc), so the bits depend neither on the device that scores the pair nor on which shard holds which row.
__global__ void __launch_bounds__(256)
pairs_rescore_kernel(const __grid_constant__ PairRows rows, int d4, const u64* __restrict__ keys, int64_t count, float* __restrict__ scores)
{
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = warp_global; c < count; c += nwarps) {
        const u64 pr = ~keys[c];
        const int64_t ri = (int64_t)(pr >> 32), rj = (int64_t)(uint32_t)pr;
        const int si = rows.shard_of(ri), sj = rows.shard_of(rj);
        const float4* pq = reinterpret_cast<const float4*>(rows.M[si]) + (ri - rows.row0[si]) * d4;
        const float4* pm = reinterpret_cast<const float4*>(rows.M[sj]) + (rj - rows.row0[sj]) * d4;
        float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
        int ch = lane;
        for (; ch + 32 < d4; ch += 64) {
            const float4 m0 = ldg_stream(pm + ch), m1 = ldg_stream(pm + ch + 32);
            const float4 q0 = ldg_stream(pq + ch), q1 = ldg_stream(pq + ch + 32);
            fma4(a0, m0, q0); fma4(a1, m1, q1);
        }
        if (ch < d4) { const float4 m0 = ldg_stream(pm + ch), q0 = ldg_stream(pq + ch); fma4(a0, m0, q0); }
        const float sc = warp_sum(((a0.x + a1.x) + (a0.y + a1.y)) + ((a0.z + a1.z) + (a0.w + a1.w)));
        if (lane == 0) scores[c] = sc;
    }
}

// out[r] = (ids[i], ids[j]) of the pair at sorted position sel[r]; ids == nullptr: the rows themselves
__global__ void pairs_emit_kernel(const int64_t* __restrict__ sel, int64_t k, const u64* __restrict__ keys, const int64_t* __restrict__ ids,
                                  int64_t* __restrict__ out_a, int64_t* __restrict__ out_b) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= k) return;
    const u64 pr = ~keys[sel[r]];
    const int64_t i = (int64_t)(pr >> 32), j = (int64_t)(uint32_t)pr;
    out_a[r] = ids ? ids[i] : i;
    out_b[r] = ids ? ids[j] : j;
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
cudaError_t launch_pairs_fill_thr(cudaStream_t st, float* thr, int b_pad, int b, const float* scalar) {
    pairs_fill_thr_kernel<<<(b_pad + 255) / 256, 256, 0, st>>>(thr, b_pad, b, scalar);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_pairs_gather(cudaStream_t st, const u64* cand, const int32_t* cand_cnt, int cand_cap, int b, int64_t q_row0,
                                int64_t m_row0, uint32_t* list_o, u64* list_pair, int64_t list_cap, unsigned long long* state) {
    if (b <= 0) return cudaSuccess;
    pairs_gather_kernel<<<b, 256, 0, st>>>(cand, cand_cnt, cand_cap, q_row0, m_row0, list_o, list_pair, list_cap, state);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_pairs_tau(cudaStream_t st, const uint32_t* list_o, const void* vals, int64_t vals_count,
                             const unsigned long long* state, int64_t list_cap, int n, float eps2, float* thr_scalar) {
    pairs_tau_kernel<<<1, PR_THREADS, 0, st>>>(list_o, reinterpret_cast<const __half*>(vals), vals_count, state, list_cap, n, eps2, thr_scalar);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_pairs_compact(cudaStream_t st, int device, const uint32_t* src_o, const u64* src_pair, const unsigned long long* src_state,
                                 int64_t list_cap, uint32_t* dst_o, u64* dst_pair, unsigned long long* dst_state, const float* thr_scalar) {
    pairs_compact_kernel<<<sm_count(device) * 4, 256, 0, st>>>(src_o, src_pair, src_state, list_cap, dst_o, dst_pair, dst_state, thr_scalar);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_pairs_sortkeys(cudaStream_t st, const u64* list_pair, int64_t count, int64_t np2, u64* keys) {
    const unsigned blocks = (unsigned)((np2 / 256 < 4096) ? (np2 / 256 > 0 ? np2 / 256 : 1) : 4096);
    pairs_sortkeys_kernel<<<blocks, 256, 0, st>>>(list_pair, count, np2, keys);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_pairs_rescore(cudaStream_t st, int device, const PairRows& rows, int ld, const u64* keys, int64_t count, float* scores) {
    if (count <= 0) return cudaSuccess;
    int64_t blocks = (count + 7) / 8;
    const int64_t cap = (int64_t)sm_count(device) * 8;
    if (blocks > cap) blocks = cap;
    pairs_rescore_kernel<<<(unsigned)blocks, 256, 0, st>>>(rows, ld / 4, keys, count, scores);
    count_launch();
    return cudaGetLastError();
}
cudaError_t launch_pairs_emit(cudaStream_t st, const int64_t* sel, int64_t k, const u64* keys, const int64_t* ids, int64_t* out_a, int64_t* out_b) {
    if (k <= 0) return cudaSuccess;
    pairs_emit_kernel<<<(unsigned)((k + 255) / 256), 256, 0, st>>>(sel, k, keys, ids, out_a, out_b);
    count_launch();
    return cudaGetLastError();
}

}  // namespace svsb
