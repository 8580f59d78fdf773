// K1 -- the similarity kernel: scores = M . q for a row-major fp32 matrix, streamed once from HBM.
//
// Replaces `x = np.dot(embeddings_matrix, query_vec)` (reference src/svs/kb.py:1185, 1623), which is
// ~97 % of the reference's warm query time and purely DRAM-bound.  Algorithmic traffic: n*d*4 bytes read
// per query (+ 4n bytes of scores written, + one 64-bit atomic per warp-iteration for the group maxima
// that seed the exact top-k, see select.cu).  No tensor cores: one query is a GEMV, 0.5 FLOP/byte.
//
// Two implementations of the same contract (kernels.cuh: launch_gemv):
//   variant 1  "ldg" : persistent grid; each warp owns R consecutive rows per iteration and issues
//                      R*U independent 128-bit streaming loads (ld.global.nc.L1::no_allocate) per lane
//                      before consuming them; query vector in shared memory; warp-shuffle reduction.
//   variant 2  "tma" : persistent grid, one CTA per SM; a producer thread streams contiguous tiles of
//                      rows into a shared-memory ring with cp.async.bulk (TMA bulk copy, UBLKCP) completing
//                      on mbarriers; consumer warps read the tile and the query from shared memory.
// Which one runs by default is decided by measurement (profiles/), not by taste.
#include "kernels.cuh"
#include <cuda_fp16.h>
#include <cstdlib>

namespace svsb {

// =============================================================================================
// variant 1: LDG.128 streaming
// =============================================================================================
template <int R, int U, int THREADS>
__global__ void __launch_bounds__(THREADS)
gemv_ldg_kernel(const float4* __restrict__ M, int64_t n, int d4, const float4* __restrict__ q,
                float* __restrict__ scores, u64* __restrict__ gmax, int group_shift, const uint8_t* __restrict__ live)
{
    extern __shared__ float4 sq[];
    pdl_wait();                                   // the query (and the scores buffer) belong to the previous kernels
    pdl_trigger();
    for (int c = threadIdx.x; c < d4; c += THREADS) sq[c] = __ldcg(q + c);   // L2 only: see gemv_tma_kernel
    __syncthreads();

    constexpr int WARPS = THREADS / 32;
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = (int64_t)blockIdx.x * WARPS + (threadIdx.x >> 5);
    const int64_t nwarps = (int64_t)gridDim.x * WARPS;
    const int64_t ngroups = (n + R - 1) / R;

    for (int64_t g = warp_global; g < ngroups; g += nwarps) {
        const int64_t r0 = g * R;
        const float4* rowp[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            int64_t rr = r0 + r; if (rr > n - 1) rr = n - 1;     // tail rows alias the last row (discarded)
            rowp[r] = M + rr * (int64_t)d4;
        }
        // K1's summation order, bit for bit the one of gemv_tma_kernel (which every exact path copies): lane l owns
        // chunks l, l+32, ...; the lane's even chunks accumulate into one float4, its odd ones into another.  a0 always
        // holds the accumulator of the NEXT chunk's parity: chunk u of an unrolled step goes to a0 when u is even, and
        // after a step of an odd number of chunks the two trade places.  The combine adds them pairwise, which commutes,
        // so it does not matter which of the two ends up holding the even chunks.
        float4 a0[R], a1[R];
#pragma unroll
        for (int r = 0; r < R; ++r) { a0[r] = make_float4(0.f, 0.f, 0.f, 0.f); a1[r] = a0[r]; }

        int c = lane;
        for (; c + 32 * (U - 1) < d4; c += 32 * U) {
            float4 m[U][R];
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int r = 0; r < R; ++r) m[u][r] = ldg_stream(rowp[r] + c + 32 * u);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const float4 qv = sq[c + 32 * u];
#pragma unroll
                for (int r = 0; r < R; ++r) fma4((u & 1) ? a1[r] : a0[r], m[u][r], qv);
            }
            if (U & 1) {
#pragma unroll
                for (int r = 0; r < R; ++r) { const float4 t = a0[r]; a0[r] = a1[r]; a1[r] = t; }
            }
        }
        for (; c < d4; c += 32) {
            float4 m[R];
#pragma unroll
            for (int r = 0; r < R; ++r) m[r] = ldg_stream(rowp[r] + c);
            const float4 qv = sq[c];
#pragma unroll
            for (int r = 0; r < R; ++r) { fma4(a0[r], m[r], qv); const float4 t = a0[r]; a0[r] = a1[r]; a1[r] = t; }
        }

        u64 kmax = 0;
        float mine = 0.f;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float s = warp_sum(((a0[r].x + a1[r].x) + (a0[r].y + a1[r].y)) + ((a0[r].z + a1[r].z) + (a0[r].w + a1[r].w)));
            if (live && r0 + r < n && !live[r0 + r]) s = dead_score();      // tombstoned row: sorts below every real score
            if (r0 + r < n) {
                u64 key = make_key(s, (uint32_t)(r0 + r));
                kmax = key > kmax ? key : kmax;
            }
            if (lane == r) mine = s;
        }
        if (lane < R && r0 + lane < n) scores[r0 + lane] = mine;
        if (lane == 0) atomicMax(&gmax[r0 >> group_shift], kmax);
    }
}

// =============================================================================================
// variant 2: TMA bulk copy ring
// =============================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}"
        :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar, u64 policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        :: "r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}

// NQ > 0: each lane keeps its NQ float4 of the query in registers (d4 <= 32 * NQ), so the only shared
// memory traffic is the row itself (one LDS.128 per 16 bytes streamed).  NQ == 0: query read from smem.
template <int CW, int NQ>
__global__ void __launch_bounds__((CW + 1) * 32, 1)
gemv_tma_kernel(const float* __restrict__ M, int64_t n, int d4, int tile_rows, int stages,
                const float* __restrict__ q, float* __restrict__ scores, u64* __restrict__ gmax, int group_shift,
                const uint8_t* __restrict__ live)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t row_bytes = (uint32_t)d4 * 16u;
    const uint32_t stage_bytes = (uint32_t)tile_rows * row_bytes;
    float4* sq = reinterpret_cast<float4*>(smem_raw + (size_t)stages * stage_bytes);   // used only when NQ == 0
    uint64_t* full = reinterpret_cast<uint64_t*>(sq + (NQ == 0 ? d4 : 0));
    uint64_t* empty = full + stages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // Programmatic dependent launch (one-query-in-flight chains): the matrix does not depend on the previous kernel, so
    // the producer starts streaming tiles at once; whoever reads the query or writes scores / group maxima waits first.
    if (NQ == 0) {
        pdl_wait();
        for (int c = threadIdx.x; c < d4; c += blockDim.x) sq[c] = __ldcg(reinterpret_cast<const float4*>(q) + c);
    }
    if (threadIdx.x == 0) {
        pdl_trigger();
        for (int s = 0; s < stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int64_t ntiles = (n + tile_rows - 1) / tile_rows;
    if (warp == CW) {
        // ---- producer: one thread streams tiles of consecutive rows (contiguous bytes) into the ring
        if (lane == 0) {
            u64 policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            int s = 0; uint32_t phase = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
                mbar_wait(&empty[s], phase ^ 1u);
                const int64_t r0 = t * tile_rows;
                const int64_t left = n - r0;
                const uint32_t rows = left < tile_rows ? (uint32_t)left : (uint32_t)tile_rows;
                const uint32_t bytes = rows * row_bytes;
                mbar_arrive_expect_tx(&full[s], bytes);
                bulk_g2s(smem_raw + (size_t)s * stage_bytes, M + r0 * (int64_t)d4 * 4, bytes, &full[s], policy);
                if (++s == stages) { s = 0; phase ^= 1u; }
            }
        }
    } else {
        // ---- consumers: warp w takes rows w, w+CW, ... of each tile
        float4 qr[NQ > 0 ? NQ : 1];
        if (NQ > 0) {
            pdl_wait();
#pragma unroll
            for (int j = 0; j < NQ; ++j) {
                const int c = lane + 32 * j;
                // ld.global.cg, not the read-only (.nc) path: under programmatic dependent launch this grid is resident
                // while the previous kernel WRITES q, which the read-only path is not allowed to observe (measured:
                // 1 query in ~1000 came out with a mixture of old and new q, scripts/pdl_stress.py)
                qr[j] = c < d4 ? __ldcg(reinterpret_cast<const float4*>(q) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        int s = 0; uint32_t phase = 0;
        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
            const int64_t r0 = t * tile_rows;
            const int64_t left = n - r0;
            const int rows = left < tile_rows ? (int)left : tile_rows;
            mbar_wait(&full[s], phase);
            const float4* tile = reinterpret_cast<const float4*>(smem_raw + (size_t)s * stage_bytes);
            u64 kmax = 0;
            for (int r = warp; r < rows; r += CW) {
                const float4* p = tile + (size_t)r * d4;
                // tombstone byte of this row (svsb_apply_mutations); issued ahead of the row's arithmetic
                const uint8_t alive = live ? __ldg(live + r0 + r) : (uint8_t)1;
                float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
                if (NQ > 0) {
                    float4 m[NQ > 0 ? NQ : 1];
#pragma unroll
                    for (int j = 0; j < NQ; ++j) {
                        const int c = lane + 32 * j;
                        m[j] = c < d4 ? p[c] : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int j = 0; j < NQ; ++j) { if (j & 1) fma4(a1, m[j], qr[j]); else fma4(a0, m[j], qr[j]); }
                } else {
                    int c = lane;
                    for (; c + 32 < d4; c += 64) { fma4(a0, p[c], sq[c]); fma4(a1, p[c + 32], sq[c + 32]); }
                    if (c < d4) fma4(a0, p[c], sq[c]);
                }
                float sc = warp_sum(((a0.x + a1.x) + (a0.y + a1.y)) + ((a0.z + a1.z) + (a0.w + a1.w)));
                if (!alive) sc = dead_score();
                if (lane == 0) {
                    scores[r0 + r] = sc;
                    const u64 k0 = make_key(sc, (uint32_t)(r0 + r));
                    kmax = k0 > kmax ? k0 : kmax;
                }
            }
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[s]);
                if (kmax) atomicMax(&gmax[r0 >> group_shift], kmax);
            }
            if (++s == stages) { s = 0; phase ^= 1u; }
        }
    }
}

// =============================================================================================
// variant 2b: the same ring, several queries per pass (small exact batches)
// =============================================================================================
// b queries against the matrix in ONE pass over HBM, bit-identical to b single-query passes: every (row, query) dot
// product is computed by one warp with exactly gemv_tma_kernel's arithmetic (lane l owns the float4 chunks l, l+32, ...;
// even chunks accumulate into a0, odd ones into a1; same combine, same xor tree).  The consumer warps are split into
// `groups` groups; a warp keeps BQ queries (its slice of each) in registers -- 4 * NQ * BQ of them, which is why the
// consumers run at 240 registers (setmaxnreg: the producer warpgroup gives its registers up) -- and the warps of a group
// share the rows of a tile.  Shared-memory traffic per streamed byte: 1 write (TMA) + `groups` reads, against ~5x
// headroom of shared-memory over HBM bandwidth per SM; the FMA pipe sees b FMAs per streamed float (b = 8: 40 %).
// Warps 0-3: producer warpgroup (one lane issues the bulk copies); warps 4-11: consumers.
// Two fp32 FMAs per instruction (Blackwell FFMA2, PTX fma.rn.f32x2): each half is an ordinary IEEE round-to-nearest FMA,
// so the bits equal two fmaf calls; what halves is the number of issue slots the b-fold arithmetic of a row needs.
struct f4x2 { u64 xy, zw; };                                    // a float4 held as two packed pairs
__device__ __forceinline__ void fma4_x2(f4x2& acc, const f4x2& a, const f4x2& b) {
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc.xy) : "l"(a.xy), "l"(b.xy));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc.zw) : "l"(a.zw), "l"(b.zw));
}
__device__ __forceinline__ f4x2 as_f4x2(const ulonglong2& v) { f4x2 r; r.xy = v.x; r.zw = v.y; return r; }
__device__ __forceinline__ float4 as_float4(const f4x2& v) {
    float4 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v.xy));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.z), "=f"(r.w) : "l"(v.zw));
    return r;
}

// FULL: d4 == 32 * NQ exactly (d = 1536, 3072, 768, 256 ...): no per-chunk bounds predicate / zero select.
template <int NQ, int BQ, bool FULL>
__global__ void __launch_bounds__(384, 1)
gemv_tma_mq_kernel(const float* __restrict__ M, int64_t n, int d4, int tile_rows, int stages,
                   const float* __restrict__ Q, int b, int groups, float* __restrict__ scores, int64_t n_stride,
                   u64* __restrict__ gmax, int64_t g_stride, int group_shift, const uint8_t* __restrict__ live)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t row_bytes = (uint32_t)d4 * 16u;
    const uint32_t stage_bytes = (uint32_t)tile_rows * row_bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)stages * stage_bytes);
    uint64_t* empty = full + stages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int CW = 8;
    if (threadIdx.x == 0) {
        for (int s = 0; s < stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t ntiles = (n + tile_rows - 1) / tile_rows;
    if (warp < 4) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == 0 && lane == 0) {
            u64 policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            int s = 0; uint32_t phase = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
                mbar_wait(&empty[s], phase ^ 1u);
                const int64_t r0 = t * tile_rows;
                const int64_t left = n - r0;
                const uint32_t rows = left < tile_rows ? (uint32_t)left : (uint32_t)tile_rows;
                const uint32_t bytes = rows * row_bytes;
                mbar_arrive_expect_tx(&full[s], bytes);
                bulk_g2s(smem_raw + (size_t)s * stage_bytes, M + r0 * (int64_t)d4 * 4, bytes, &full[s], policy);
                if (++s == stages) { s = 0; phase ^= 1u; }
            }
        }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 240;");
        const int cw = warp - 4, grp = cw % groups, sub = cw / groups, nsub = CW / groups;
        f4x2 qr[BQ][NQ];
#pragma unroll
        for (int u = 0; u < BQ; ++u) {
            int qi = grp * BQ + u;
            if (qi > b - 1) qi = b - 1;                          // padding slots recompute the last query; never stored
            const ulonglong2* qp = reinterpret_cast<const ulonglong2*>(Q) + (int64_t)qi * d4;
#pragma unroll
            for (int j = 0; j < NQ; ++j) {
                const int c = lane + 32 * j;
                qr[u][j] = as_f4x2((FULL || c < d4) ? __ldcg(qp + c) : make_ulonglong2(0ull, 0ull));
            }
        }
        int s = 0; uint32_t phase = 0;
        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
            const int64_t r0 = t * tile_rows;
            const int64_t left = n - r0;
            const int rows = left < tile_rows ? (int)left : tile_rows;
            mbar_wait(&full[s], phase);
            const ulonglong2* tile = reinterpret_cast<const ulonglong2*>(smem_raw + (size_t)s * stage_bytes);
            for (int r = sub; r < rows; r += nsub) {
                const ulonglong2* p = tile + (size_t)r * d4;
                const uint8_t alive = live ? __ldg(live + r0 + r) : (uint8_t)1;
                f4x2 a0[BQ], a1[BQ];
#pragma unroll
                for (int u = 0; u < BQ; ++u) { a0[u].xy = 0ull; a0[u].zw = 0ull; a1[u] = a0[u]; }
                // With 192 registers of queries there is no room to load the whole row slice ahead of the arithmetic (as
                // the single-query kernel does): keep PF loads in flight instead, issued a chunk ahead of their FMAs --
                // without it every chunk pays a shared-memory round trip with only two warps per scheduler to hide it
                // (measured: 2.1 ms instead of 1.0 ms for 8 queries at 1M x 1536).
                constexpr int PF = (4 * NQ * BQ >= 192) ? 2 : NQ;
                ulonglong2 mb[PF];
#pragma unroll
                for (int j = 0; j < PF && j < NQ; ++j) { const int c = lane + 32 * j; mb[j] = (FULL || c < d4) ? p[c] : make_ulonglong2(0ull, 0ull); }
#pragma unroll
                for (int j = 0; j < NQ; ++j) {
                    const f4x2 m = as_f4x2(mb[j % PF]);
                    if (j + PF < NQ) { const int c = lane + 32 * (j + PF); mb[j % PF] = (FULL || c < d4) ? p[c] : make_ulonglong2(0ull, 0ull); }
#pragma unroll
                    for (int u = 0; u < BQ; ++u) { if (j & 1) fma4_x2(a1[u], m, qr[u][j]); else fma4_x2(a0[u], m, qr[u][j]); }
                }
                // the BQ xor trees advance in lockstep (BQ independent shuffles per round instead of BQ serial trees), then
                // lane u publishes query u: one predicated block of stores for the whole row
                float v[BQ];
#pragma unroll
                for (int u = 0; u < BQ; ++u) {
                    const float4 x0 = as_float4(a0[u]), x1 = as_float4(a1[u]);
                    v[u] = ((x0.x + x1.x) + (x0.y + x1.y)) + ((x0.z + x1.z) + (x0.w + x1.w));
                }
                // BQ xor trees in one: at distance 16 a lane keeps the upper or the lower half of the queries and trades the
                // other half with its partner, at distance 8 a quarter, ... -- every addition is still x[l] + x[l ^ o] of ONE
                // query at the distances 16, 8, 4, 2, 1 in that order, i.e. exactly warp_sum's tree (fp32 addition is
                // commutative bit for bit), with 2*BQ - 2 + log2(32 / BQ) shuffles instead of 5 * BQ.
                int o = 16;
#pragma unroll
                for (int cnt = BQ; cnt > 1; cnt >>= 1, o >>= 1) {
                    const int half = cnt >> 1;
                    const bool up = (lane & o) != 0;
#pragma unroll
                    for (int i = 0; i < half; ++i) {
                        const float send = up ? v[i] : v[i + half];
                        const float keep = up ? v[i + half] : v[i];
                        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                    }
                }
#pragma unroll
                for (; o > 0; o >>= 1) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
                float sc = v[0];                                 // the sum of query u_of(lane), complete in every lane
                if (!alive) sc = dead_score();
                // which query this lane holds: bit 4 picked a half, bit 3 a quarter, ...; lanes with the low bits clear publish
                constexpr int LANES_PER_Q = 32 / BQ;
                int u_mine = 0;
#pragma unroll
                for (int step = 0, bit = 16, w = BQ >> 1; w >= 1; ++step, bit >>= 1, w >>= 1) u_mine += (lane & bit) ? w : 0;
                const int qi = grp * BQ + u_mine;
                if ((lane & (LANES_PER_Q - 1)) == 0 && qi < b) {
                    scores[(int64_t)qi * n_stride + r0 + r] = sc;
                    atomicMax(&gmax[(int64_t)qi * g_stride + ((r0 + r) >> group_shift)], make_key(sc, (uint32_t)(r0 + r)));
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (++s == stages) { s = 0; phase ^= 1u; }
        }
    }
}

// =============================================================================================
// variant 3: the int8 filter -- the same ring over the int8 shadow, then an exact re-score of the few candidates
// =============================================================================================
// A single query reads n*d*4 bytes with K1 at the HBM rate; the filter reads the int8 shadow instead (n*ld8 bytes plus
// 4n for the row scales) and writes K1's outputs -- scores[n], group maxima -- as COARSE values.  filter_threshold_kernel
// turns them into a threshold T <= tau~ - 2 eps (tau~ = the kk-th largest coarse score), filter_rescore_kernel gives
// every row with coarse >= T its exact score (K1's arithmetic, bit for bit) and every other row of the groups it rescans
// the tombstone score, and rewrites the group maxima so that the unchanged selection kernel sees only exact scores.
// Exactness (DESIGN.md section 4, "K1f8"): |coarse - exact| <= eps, kk rows have coarse >= tau~, so every row of the
// exact top-kk has coarse >= tau~ - 2 eps >= T.
//
// Row r of the shadow is Q_r[ld8] (int8, zero padded) with one fp32 scale s_r = max|r_j| / 127: r^ = s_r * Q_r.  The
// device word E >= max_r ||r - r^|| bounds the quantisation error of every row converted so far (it only grows).  The
// query is split into two int8 terms q^ = s1 * q_hi + s2 * q_lo (s1 = max|q_j| / 127, s2 = s1 / 254) by q8_split, the
// same function in the pass and in the threshold kernel, so both see the same bits; each row is two exact int32 dp4a
// sums and one fp32 combine, coarse = s_r * (s1 * D_hi + s2 * D_lo).  The bound is in filter_threshold_kernel.
__device__ __forceinline__ int q8_round(float x) { return max(-127, min(127, __float2int_rn(x))); }
// |x| as bits: unsigned order is the order of non-negative floats, NaN above +inf (the same maximum in any order)
__device__ __forceinline__ uint32_t abs_bits(float x) { return __float_as_uint(x) & 0x7fffffffu; }
__device__ __forceinline__ void q8_scales(uint32_t amax_bits, float& s1, float& s2) {
    s1 = __fdiv_rn(__uint_as_float(amax_bits), 127.f);
    s2 = __fdiv_rn(s1, 254.f);
}
// s1 == 0 (a zero query) divides by nothing; a non-finite query gives some q_hi / q_lo and its threshold takes every row
__device__ __forceinline__ void q8_split(float v, float s1, float s2, int& hi, int& lo) {
    hi = s1 > 0.f ? q8_round(__fdiv_rn(v, s1)) : 0;
    const float res = fmaf(-s1, (float)hi, v);
    lo = s2 > 0.f ? q8_round(__fdiv_rn(res, s2)) : 0;
}

// One warp per row: scale8[r], M8[r][0..ld8), and E raised to this row's ||r - r^|| (computed in double, rounded up).
__global__ void __launch_bounds__(256)
rows_to_i8_kernel(const float* __restrict__ M, int64_t n, int ld, int8_t* __restrict__ M8, int ld8, float* __restrict__ scale8,
                  uint32_t* __restrict__ emax)
{
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < n; r += nwarps) {
        const float4* row = reinterpret_cast<const float4*>(M + r * (int64_t)ld);
        uint32_t mb = 0u;
        for (int c = lane; c < ld / 4; c += 32) {
            const float4 v = __ldg(row + c);
            mb = max(max(mb, abs_bits(v.x)), max(abs_bits(v.y), max(abs_bits(v.z), abs_bits(v.w))));
        }
        mb = __reduce_max_sync(0xffffffffu, mb);
        const float s = __fdiv_rn(__uint_as_float(mb), 127.f);
        double e2 = 0.0;
        for (int c = lane; c < ld8 / 4; c += 32) {
            const float4 v = 4 * c < ld ? __ldg(row + c) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float x[4] = {v.x, v.y, v.z, v.w};
            uint32_t packed = 0u;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int qv = s > 0.f ? q8_round(__fdiv_rn(x[t], s)) : 0;
                const double err = (double)x[t] - (double)s * (double)qv;          // s * qv is exact in double
                e2 = fma(err, err, e2);
                packed |= (uint32_t)(qv & 0xff) << (8 * t);
            }
            reinterpret_cast<uint32_t*>(M8 + r * (int64_t)ld8)[c] = packed;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, o);
        if (lane == 0) {
            scale8[r] = s;
            atomicMax(emax, __float_as_uint(__double2float_ru(sqrt(e2) * (1.0 + 1.0 / 1048576.0))));
        }
    }
}

// One row's two dp4a sums over the lane's NC chunks, each split into two partial accumulators (x, y words and z, w
// words): integer sums are exact in any order, so the split halves the dependent chain without changing a bit.
template <int NC>
__device__ __forceinline__ void dot8(const uint4 (&m)[NC], const uint32_t (&qh)[NC][4], const uint32_t (&ql)[NC][4], int& dh, int& dl) {
    int h0 = 0, h1 = 0, l0 = 0, l1 = 0;                      // |sum| <= 3072 * 127^2 < 2^31: exact
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        h0 = __dp4a((int)m[j].x, (int)qh[j][0], h0); l0 = __dp4a((int)m[j].x, (int)ql[j][0], l0);
        h1 = __dp4a((int)m[j].z, (int)qh[j][2], h1); l1 = __dp4a((int)m[j].z, (int)ql[j][2], l1);
        h0 = __dp4a((int)m[j].y, (int)qh[j][1], h0); l0 = __dp4a((int)m[j].y, (int)ql[j][1], l0);
        h1 = __dp4a((int)m[j].w, (int)qh[j][3], h1); l1 = __dp4a((int)m[j].w, (int)ql[j][3], l1);
    }
    dh = h0 + h1; dl = l0 + l1;
}

// Shared memory of gemv8_tma_kernel behind the ring of `stages` tiles: per stage a side slot (the tile's row scales,
// then its tombstone bytes), then the query's two int8 terms, the consumer warps' maxima of |q_j| and the barriers.
// tile_rows % 16 == 0 keeps every part 16-byte aligned.
__host__ __device__ constexpr size_t filter8_side_bytes(int tile_rows) { return (size_t)tile_rows * 5; }
__host__ __device__ constexpr size_t filter8_smem_bytes(int tile_rows, int stages, int ld8) {
    return (size_t)stages * ((size_t)tile_rows * ld8 + filter8_side_bytes(tile_rows)) + 2 * (size_t)ld8 + 64 + (size_t)stages * 16;
}

// NC: 16-byte chunks (16 int8) of the shadow row per lane, c8 = ld8 / 16 <= 32 * NC.  The query's two int8 terms stay in
// registers (2 * NC uint4).  No element is widened to fp32: per row 8 * NC dp4a per lane, two warp reductions, one combine.
// The producer stages each tile's row scales (and tombstone bytes) through the ring with the rows, so the consumers'
// tile loop reads shared memory only; a consumer warp works on two rows of a tile at once (w and w + CW) to overlap
// their shared-memory loads, dp4a chains and reductions.
template <int CW, int NC>
__global__ void __launch_bounds__((CW + 1) * 32, 1)
gemv8_tma_kernel(const int8_t* __restrict__ M8, const float* __restrict__ scale8, int64_t n, int c8, int tile_rows, int stages,
                 const float* __restrict__ q, int ld, float* __restrict__ scores, u64* __restrict__ gmax, int group_shift,
                 const uint8_t* __restrict__ live)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const uint32_t row_bytes = (uint32_t)c8 * 16u;
    const uint32_t stage_bytes = (uint32_t)tile_rows * row_bytes;
    const uint32_t side_bytes = (uint32_t)filter8_side_bytes(tile_rows);
    unsigned char* side = smem_raw + (size_t)stages * stage_bytes;
    uint32_t* sqh = reinterpret_cast<uint32_t*>(side + (size_t)stages * side_bytes);   // c8 * 4 words each
    uint32_t* sql = sqh + 4 * c8;
    uint32_t* samax = sql + 4 * c8;                                                      // CW <= 16 words
    uint64_t* full = reinterpret_cast<uint64_t*>(samax + 16);
    uint64_t* empty = full + stages;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        pdl_trigger();
        for (int s = 0; s < stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], CW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int64_t ntiles = (n + tile_rows - 1) / tile_rows;
    if (warp == CW) {
        if (lane == 0) {
            u64 policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            int s = 0; uint32_t phase = 0;
            for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
                mbar_wait(&empty[s], phase ^ 1u);
                const int64_t r0 = t * tile_rows;
                const int64_t left = n - r0;
                const uint32_t rows = left < tile_rows ? (uint32_t)left : (uint32_t)tile_rows;
                const uint32_t bytes = rows * row_bytes;
                // bulk copies move multiples of 16 bytes: the scales are read up to round_up(n, 4) (inside the shadow's
                // allocation: its E word follows them), the tombstone bytes up to round_up(n, 16) (svsb_apply_mutations
                // allocates that much); the rounded tails land in the side slot and are never read
                const uint32_t sbytes = ((rows + 3u) & ~3u) * 4u, lbytes = live ? (rows + 15u) & ~15u : 0u;
                unsigned char* sd = side + (size_t)s * side_bytes;
                mbar_arrive_expect_tx(&full[s], bytes + sbytes + lbytes);
                bulk_g2s(smem_raw + (size_t)s * stage_bytes, reinterpret_cast<const unsigned char*>(M8) + (size_t)r0 * row_bytes,
                         bytes, &full[s], policy);
                bulk_g2s(sd, scale8 + r0, sbytes, &full[s], policy);
                if (live) bulk_g2s(sd + 4 * tile_rows, live + r0, lbytes, &full[s], policy);
                if (++s == stages) { s = 0; phase ^= 1u; }
            }
        }
    } else {
        // The query's split, once per CTA: consumer thread i converts words i, i + 32 CW, ... (4 components each) of
        // the c8 * 4; the maximum of |q_j| is reduced over the consumer warps first (a named barrier: the producer
        // does not join).  q8_scales / q8_split are the threshold kernel's, so both see the same bits.
        pdl_wait();                                   // the query is written by the previous kernel (see gemv_tma_kernel)
        constexpr int QW = (128 * NC + 32 * CW - 1) / (32 * CW);      // words per consumer thread
        const int ct = threadIdx.x, nw = 4 * c8, ld4 = ld >> 2;
        float4 qv[QW];
        uint32_t mb = 0u;
#pragma unroll
        for (int i = 0; i < QW; ++i) {
            const int w = ct + 32 * CW * i;
            qv[i] = w < ld4 ? __ldcg(reinterpret_cast<const float4*>(q) + w) : make_float4(0.f, 0.f, 0.f, 0.f);
            mb = max(max(mb, abs_bits(qv[i].x)), max(abs_bits(qv[i].y), max(abs_bits(qv[i].z), abs_bits(qv[i].w))));
        }
        mb = __reduce_max_sync(0xffffffffu, mb);
        if (lane == 0) samax[warp] = mb;
        asm volatile("bar.sync 1, %0;" :: "n"(CW * 32) : "memory");
#pragma unroll
        for (int w = 0; w < CW; ++w) mb = max(mb, samax[w]);
        float s1, s2;
        q8_scales(mb, s1, s2);
#pragma unroll
        for (int i = 0; i < QW; ++i) {
            const int w = ct + 32 * CW * i;
            if (w < nw) {
                const float x[4] = {qv[i].x, qv[i].y, qv[i].z, qv[i].w};
                uint32_t h = 0u, l = 0u;
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    int hi, lo;
                    q8_split(x[b], s1, s2, hi, lo);
                    h |= (uint32_t)(hi & 0xff) << (8 * b);
                    l |= (uint32_t)(lo & 0xff) << (8 * b);
                }
                sqh[w] = h; sql[w] = l;
            }
        }
        asm volatile("bar.sync 1, %0;" :: "n"(CW * 32) : "memory");
        // lane l's chunks l, l + 32, ... are query components [16c, 16c + 16)
        uint32_t qh[NC][4], ql[NC][4];
#pragma unroll
        for (int j = 0; j < NC; ++j) {
            const int c = lane + 32 * j;
            const uint4 h = c < c8 ? reinterpret_cast<const uint4*>(sqh)[c] : make_uint4(0u, 0u, 0u, 0u);
            const uint4 l = c < c8 ? reinterpret_cast<const uint4*>(sql)[c] : make_uint4(0u, 0u, 0u, 0u);
            qh[j][0] = h.x; qh[j][1] = h.y; qh[j][2] = h.z; qh[j][3] = h.w;
            ql[j][0] = l.x; ql[j][1] = l.y; ql[j][2] = l.z; ql[j][3] = l.w;
        }
        int s = 0; uint32_t phase = 0;
        for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
            const int64_t r0 = t * tile_rows;
            const int64_t left = n - r0;
            const int rows = left < tile_rows ? (int)left : tile_rows;
            mbar_wait(&full[s], phase);
            const uint4* tile = reinterpret_cast<const uint4*>(smem_raw + (size_t)s * stage_bytes);
            const float* ssc = reinterpret_cast<const float*>(side + (size_t)s * side_bytes);
            const uint8_t* slive = side + (size_t)s * side_bytes + 4 * tile_rows;
            u64 kmax = 0;
            for (int ra = warp; ra < rows; ra += 2 * CW) {
                // rows ra and rb = ra + CW together; a missing rb (odd count, partial tile) repeats ra and is not stored
                const int rb = ra + CW < rows ? ra + CW : ra;
                const uint4* pa = tile + (size_t)ra * c8;
                const uint4* pb = tile + (size_t)rb * c8;
                uint4 ma[NC], mbv[NC];
#pragma unroll
                for (int j = 0; j < NC; ++j) {
                    const int c = lane + 32 * j;
                    ma[j] = c < c8 ? pa[c] : make_uint4(0u, 0u, 0u, 0u);
                    mbv[j] = c < c8 ? pb[c] : make_uint4(0u, 0u, 0u, 0u);
                }
                int dha, dla, dhb, dlb;
                dot8<NC>(ma, qh, ql, dha, dla);
                dot8<NC>(mbv, qh, ql, dhb, dlb);
                dha = __reduce_add_sync(0xffffffffu, dha);
                dla = __reduce_add_sync(0xffffffffu, dla);
                dhb = __reduce_add_sync(0xffffffffu, dhb);
                dlb = __reduce_add_sync(0xffffffffu, dlb);
                float sca = ssc[ra] * fmaf(s2, (float)dla, s1 * (float)dha);
                float scb = ssc[rb] * fmaf(s2, (float)dlb, s1 * (float)dhb);
                if (live) {
                    if (!slive[ra]) sca = dead_score();
                    if (!slive[rb]) scb = dead_score();
                }
                if (lane == 0) {
                    scores[r0 + ra] = sca;
                    const u64 ka = make_key(sca, (uint32_t)(r0 + ra));
                    kmax = ka > kmax ? ka : kmax;
                    if (rb != ra) {
                        scores[r0 + rb] = scb;
                        const u64 kb = make_key(scb, (uint32_t)(r0 + rb));
                        kmax = kb > kmax ? kb : kmax;
                    }
                }
            }
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&empty[s]);
                if (kmax) atomicMax(&gmax[r0 >> group_shift], kmax);
            }
            if (++s == stages) { s = 0; phase ^= 1u; }
        }
    }
}

// One CTA.  state[0] = T as an ordered key word (f32_to_ordered): the rows with f32_to_ordered(coarse) >= T are the
// candidates; T = 0 takes every row (no usable threshold: at most kk groups, a non-finite query, bound or group maximum).
// state[1] = 0 (the re-score kernel counts its rows there).
// T = (kk-th largest group maximum) - 2 eps, rounded down: that maximum comes from kk distinct rows, so it is <= tau~.
// eps bounds |coarse - exact| (DESIGN.md section 4, "K1f8"): with e8 = the int8 shadow's E, R = max_row_norm,
// R^ = R + E >= max ||r^||, q^ from q8_split, eps = ||q|| E + ||q - q^|| R^ + ld 2^-23 ||q|| R (K1's fp32 sum)
// + 2^-21 (||s1 q_hi|| + ||s2 q_lo||) R^ (the combine's five roundings), times 1 + 2^-10 for the fp32 norms, + 1e-8.
constexpr int FT_THREADS = 1024;
constexpr int FT_PER_THREAD = (int)(GROUPS_TARGET / FT_THREADS);
__global__ void __launch_bounds__(FT_THREADS, 1)
filter_threshold_kernel(const u64* __restrict__ gmax, int G, int kk, const float* __restrict__ q, int ld,
                        float max_row_norm, const float* __restrict__ e8, uint32_t* __restrict__ state)
{
    __shared__ uint32_t hist[256];
    __shared__ float red[FT_THREADS / 32];
    __shared__ uint32_t amx[FT_THREADS / 32];
    __shared__ double red8[3][FT_THREADS / 32];
    __shared__ uint32_t sh_prefix, sh_want;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float ss = 0.f;
    uint32_t mb = 0u;
    for (int i = tid; i < ld; i += FT_THREADS) { const float v = __ldcg(q + i); ss = fmaf(v, v, ss); mb = max(mb, abs_bits(v)); }
    ss = warp_sum(ss);
    if (lane == 0) red[warp] = ss;
    mb = __reduce_max_sync(0xffffffffu, mb);
    if (lane == 0) amx[warp] = mb;
    uint32_t v[FT_PER_THREAD];                         // high words of the group maxima (ordered coarse scores)
#pragma unroll
    for (int j = 0; j < FT_PER_THREAD; ++j) { const int i = tid + j * FT_THREADS; v[j] = i < G ? (uint32_t)(__ldcg(gmax + i) >> 32) : 0u; }
    if (tid == 0) { sh_prefix = 0u; sh_want = (uint32_t)kk; }
    __syncthreads();
    {                                                  // ||q - q^||^2, ||s1 q_hi||^2, ||s2 q_lo||^2 (double: exact enough)
        for (int w = 0; w < FT_THREADS / 32; ++w) mb = max(mb, amx[w]);
        float s1, s2;
        q8_scales(mb, s1, s2);
        double a[3] = {0.0, 0.0, 0.0};
        for (int i = tid; i < ld; i += FT_THREADS) {
            const float x = __ldcg(q + i);
            int hi, lo;
            q8_split(x, s1, s2, hi, lo);
            const double th = (double)s1 * hi, tl = (double)s2 * lo, r = (double)x - th - tl;
            a[0] = fma(r, r, a[0]); a[1] = fma(th, th, a[1]); a[2] = fma(tl, tl, a[2]);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a[c] += __shfl_xor_sync(0xffffffffu, a[c], o);
            if (lane == 0) red8[c][warp] = a[c];
        }
    }
    // kk-th largest of the G words: radix select, 8 bits per round from the top
    uint32_t mask = 0u;
    for (int shift = 24; shift >= 0; shift -= 8) {
        if (tid < 256) hist[tid] = 0u;
        __syncthreads();
        const uint32_t prefix = sh_prefix;
#pragma unroll
        for (int j = 0; j < FT_PER_THREAD; ++j)
            if (tid + j * FT_THREADS < G && (v[j] & mask) == prefix) atomicAdd(&hist[(v[j] >> shift) & 255u], 1u);
        __syncthreads();
        if (warp == 0) {
            // lane l owns bins [8l, 8l + 8); suffix[l] = entries in bins >= 8l
            uint32_t c = 0;
#pragma unroll
            for (int b = 0; b < 8; ++b) c += hist[8 * lane + b];
            uint32_t suf = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_down_sync(0xffffffffu, suf, o); if (lane + o < 32) suf += t; }
            const uint32_t want = sh_want;
            const unsigned ball = __ballot_sync(0xffffffffu, suf >= want);
            const int top = 31 - __clz(ball);              // the highest lane whose bins reach the kk-th entry
            if (lane == top) {
                uint32_t cum = suf - c;
                for (int b = 7; b >= 0; --b) {
                    const uint32_t h = hist[8 * lane + b];
                    if (cum + h >= want) { sh_prefix = prefix | ((uint32_t)(8 * lane + b) << shift); sh_want = want - cum; break; }
                    cum += h;
                }
            }
        }
        mask |= 255u << shift;
        __syncthreads();
    }
    if (tid == 0) {
        float qq = 0.f;
        for (int w = 0; w < FT_THREADS / 32; ++w) qq += red[w];
        const float qn = sqrtf(qq);
        const float tau = ordered_to_f32(sh_prefix);
        uint32_t T = 0u;
        double a[3] = {0.0, 0.0, 0.0};
        for (int w = 0; w < FT_THREADS / 32; ++w) for (int c = 0; c < 3; ++c) a[c] += red8[c][w];
        const double E = (double)__ldcg(e8), R = (double)max_row_norm, Rh = R + E;
        const double sum = (double)qn * E + sqrt(a[0]) * Rh + (double)ld * 0x1p-23 * (double)qn * R
                           + 0x1p-21 * (sqrt(a[1]) + sqrt(a[2])) * Rh;
        const double eps = __dadd_rn(__dmul_rn(sum, 1.0 + 0x1p-10), 1e-8);   // two roundings, not one fused multiply-add
        if (G > kk && isfinite(tau) && isfinite(qn) && isfinite(eps)) {
            float t = __double2float_rd((double)tau - 2.0 * eps);
            if (t == 0.f) t = -0.f;                         // f32_to_ordered(-0) < f32_to_ordered(+0): keep both zeros
            T = f32_to_ordered(t);
        }
        state[0] = T;
        state[1] = 0u;
    }
}

// One warp per row group (grid-stride).  A group whose coarse maximum reaches T: every candidate row (live, coarse >= T)
// is re-scored by the warp with gemv_tma_kernel's arithmetic (lane l owns float4 chunks l, l+32, ...; even chunks into
// a0, odd ones into a1; same combine, same xor tree) -- the bits K1 would have written; the group's other rows get the
// tombstone score; its maximum becomes the largest key over both.  Any other group's maximum becomes 0, so the
// selection kernel (which rescans only groups whose maximum reaches its kk-th largest, a candidate's key: at least kk
// groups hold a candidate) never reads its coarse scores.
template <int NQ>
__global__ void __launch_bounds__(256)
filter_rescore_kernel(const float* __restrict__ M, int64_t n, int d4, const float* __restrict__ q, float* __restrict__ scores,
                      u64* __restrict__ gmax, int group_shift, const uint8_t* __restrict__ live, uint32_t* __restrict__ state)
{
    __shared__ float4 sq[32 * NQ];
    for (int c = threadIdx.x; c < 32 * NQ; c += blockDim.x) sq[c] = c < d4 ? __ldcg(reinterpret_cast<const float4*>(q) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    __syncthreads();
    const uint32_t T = __ldcg(state);
    const int lane = threadIdx.x & 31;
    const int64_t G = (n + ((int64_t)1 << group_shift) - 1) >> group_shift;
    const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < G; g += nwarps) {
        const u64 gm = gmax[g];
        u64 kmax = 0;
        if ((uint32_t)(gm >> 32) >= T) {
            const int64_t r_beg = g << group_shift;
            const int64_t r_end = min(n, r_beg + ((int64_t)1 << group_shift));
            int found = 0;
            for (int64_t rb = r_beg; rb < r_end; rb += 32) {
                const int64_t r = rb + lane;
                const bool in = r < r_end;
                const bool alive = in && (!live || live[r]);
                const bool cand = alive && f32_to_ordered(scores[r]) >= T;
                if (in && !cand) {
                    scores[r] = dead_score();
                    const u64 k0 = make_key(dead_score(), (uint32_t)r);
                    kmax = k0 > kmax ? k0 : kmax;
                }
                unsigned ball = __ballot_sync(0xffffffffu, cand);
                found += __popc(ball);
                while (ball) {
                    const int b = __ffs(ball) - 1;
                    ball &= ball - 1;
                    const int64_t rr = rb + b;
                    const float4* p = reinterpret_cast<const float4*>(M) + rr * (int64_t)d4;
                    float4 m[NQ];
#pragma unroll
                    for (int j = 0; j < NQ; ++j) { const int c = lane + 32 * j; m[j] = c < d4 ? ldg_stream(p + c) : make_float4(0.f, 0.f, 0.f, 0.f); }
                    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0;
#pragma unroll
                    for (int j = 0; j < NQ; ++j) { if (j & 1) fma4(a1, m[j], sq[lane + 32 * j]); else fma4(a0, m[j], sq[lane + 32 * j]); }
                    const float sc = warp_sum(((a0.x + a1.x) + (a0.y + a1.y)) + ((a0.z + a1.z) + (a0.w + a1.w)));
                    if (lane == b) scores[rr] = sc;
                    const u64 k0 = make_key(sc, (uint32_t)rr);
                    kmax = k0 > kmax ? k0 : kmax;
                }
            }
            kmax = warp_max_u64(kmax);
            if (lane == 0 && found) atomicAdd(state + 1, (uint32_t)found);
        }
        if (lane == 0) gmax[g] = kmax;
    }
}

// =============================================================================================
// host side
// =============================================================================================
int sm_count(int device) {
    static int cache[64] = {0};
    if (device < 0 || device >= 64) device = 0;
    if (cache[device] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || v <= 0) v = 148;
        cache[device] = v;
    }
    return cache[device];
}

template <int R, int U, int THREADS>
static cudaError_t run_ldg(cudaStream_t st, int device, const float* M, int64_t n, int d4, const float* q,
                           float* scores, u64* gmax, int group_shift, const uint8_t* live, int blocks_per_sm)
{
    auto kern = gemv_ldg_kernel<R, U, THREADS>;
    const size_t smem = (size_t)d4 * 16;
    static thread_local int configured_dev = -1;   // opt-in to >48 KB dynamic smem (d > 3072)
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    (void)configured_dev;
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, THREADS, smem);
    if (e != cudaSuccess) return e;
    if (occ < 1) occ = 1;
    if (blocks_per_sm > 0 && blocks_per_sm < occ) occ = blocks_per_sm;
    constexpr int WARPS = THREADS / 32;
    const int64_t ngroups = (n + R - 1) / R;
    int64_t grid = (int64_t)sm_count(device) * occ;
    const int64_t need = (ngroups + WARPS - 1) / WARPS;
    if (grid > need) grid = need;
    if (grid < 1) grid = 1;
    e = launch_kernel(kern, dim3((unsigned)grid), dim3(THREADS), smem, st, reinterpret_cast<const float4*>(M), n, d4,
                      reinterpret_cast<const float4*>(q), scores, gmax, group_shift, live);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
}

template <int CW, int NQ>
static cudaError_t run_tma_inst(cudaStream_t st, int64_t grid, size_t smem, const float* M, int64_t n, int d4,
                                int tile_rows, int stages, const float* q, float* scores, u64* gmax, int group_shift,
                                const uint8_t* live)
{
    auto kern = gemv_tma_kernel<CW, NQ>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = launch_kernel(kern, dim3((unsigned)grid), dim3((CW + 1) * 32), smem, st, M, n, d4, tile_rows, stages, q, scores, gmax, group_shift, live);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
}

// tile_rows / stages: 0 = default.  cw: consumer warps (8 or 16; 0 = default).
static cudaError_t run_tma(cudaStream_t st, int device, const float* M, int64_t n, int d4, const float* q,
                           float* scores, u64* gmax, int group_shift, const uint8_t* live, int tile_rows, int stages, int cw,
                           int reserve_sms)
{
    const size_t row_bytes = (size_t)d4 * 16;
    const int nq = d4 <= 64 ? 2 : d4 <= 192 ? 6 : d4 <= 384 ? 12 : d4 <= 768 ? 24 : 0;
    const size_t q_bytes = nq == 0 ? row_bytes : 0;
    const size_t budget = 224 * 1024 - q_bytes - 256;       // ring bytes available next to q + barriers
    // Measured on B200 (profiles/r01_tune_gemv.md): ~48 KB tiles x 3 stages (~144 KB in flight per SM) is
    // the optimum; deeper rings are SLOWER (more concurrent DRAM streams), shallower ones starve.
    if (tile_rows <= 0) {
        tile_rows = 64;                                       // power of two <= 64
        while (tile_rows > 1 && (size_t)tile_rows * row_bytes > 48 * 1024) tile_rows >>= 1;
    }
    if (stages <= 0) {
        stages = (int)(budget / ((size_t)tile_rows * row_bytes));
        if (stages > 3) stages = 3;
    }
    if (tile_rows > 64 || (tile_rows & (tile_rows - 1))) return cudaErrorInvalidConfiguration;
    if (stages < 2 || stages > 16 || (size_t)stages * tile_rows * row_bytes > budget) return cudaErrorInvalidConfiguration;
    const size_t smem = (size_t)stages * tile_rows * row_bytes + q_bytes + (size_t)stages * 16 + 64;
    const int64_t ntiles = (n + tile_rows - 1) / tile_rows;
    int64_t grid = sm_count(device) - reserve_sms;          // reserve_sms: SMs left free for a concurrent selection kernel
    if (grid > ntiles) grid = ntiles;
    if (grid < 1) grid = 1;
#define SVSB_TMA_CASE(CWV, NQV) \
    return run_tma_inst<CWV, NQV>(st, grid, smem, M, n, d4, tile_rows, stages, q, scores, gmax, group_shift, live)
    if (cw == 16) {
        switch (nq) { case 2: SVSB_TMA_CASE(16, 2); case 6: SVSB_TMA_CASE(16, 6); case 12: SVSB_TMA_CASE(16, 12);
                      case 24: SVSB_TMA_CASE(16, 24); default: SVSB_TMA_CASE(16, 0); }
    }
    switch (nq) { case 2: SVSB_TMA_CASE(8, 2); case 6: SVSB_TMA_CASE(8, 6); case 12: SVSB_TMA_CASE(8, 12);
                  case 24: SVSB_TMA_CASE(8, 24); default: SVSB_TMA_CASE(8, 0); }
#undef SVSB_TMA_CASE
}

// Force the (lazily loaded) similarity kernels onto the device now.  With CUDA's lazy module loading the FIRST launch
// of a kernel synchronises the context; issued while another engine of this process has a merge kernel spinning on a
// peer flag, that first launch would wait for the spin to end -- which may be waiting for this very launch.
cudaError_t preload_gemv_kernels()
{
    cudaFuncAttributes a;
    cudaError_t e = cudaSuccess;
#define SVSB_PRE(K) do { if (e == cudaSuccess) e = cudaFuncGetAttributes(&a, K); } while (0)
    SVSB_PRE((gemv_tma_kernel<8, 2>)); SVSB_PRE((gemv_tma_kernel<8, 6>)); SVSB_PRE((gemv_tma_kernel<8, 12>));
    SVSB_PRE((gemv_tma_kernel<8, 24>)); SVSB_PRE((gemv_tma_kernel<8, 0>));
    SVSB_PRE((gemv_tma_kernel<16, 2>)); SVSB_PRE((gemv_tma_kernel<16, 6>)); SVSB_PRE((gemv_tma_kernel<16, 12>));
    SVSB_PRE((gemv_tma_kernel<16, 24>)); SVSB_PRE((gemv_tma_kernel<16, 0>));
    SVSB_PRE((gemv_ldg_kernel<4, 3, 256>));
    SVSB_PRE((gemv8_tma_kernel<8, 1>)); SVSB_PRE((gemv8_tma_kernel<8, 2>)); SVSB_PRE((gemv8_tma_kernel<8, 3>));
    SVSB_PRE((gemv8_tma_kernel<8, 4>)); SVSB_PRE((gemv8_tma_kernel<8, 6>));
    SVSB_PRE(filter_threshold_kernel);
    SVSB_PRE((filter_rescore_kernel<2>)); SVSB_PRE((filter_rescore_kernel<6>)); SVSB_PRE((filter_rescore_kernel<12>));
    SVSB_PRE((filter_rescore_kernel<24>));
#undef SVSB_PRE
    return e;
}

cudaError_t launch_gemv(cudaStream_t st, int device, const float* M, int64_t n, int d, int ld,
                        const float* q, float* scores, u64* gmax, int group_shift,
                        int variant, int tune_a, int tune_b, int reserve_sms, const uint8_t* live)
{
    (void)d;
    if (n <= 0) return cudaSuccess;
    const int d4 = ld / 4;
    if (variant == 0) {
        // rows longer than a TMA stage can hold fall back to the LDG kernel
        variant = ((size_t)d4 * 16 * 4 <= 200 * 1024) ? 2 : 1;
        // tuning knobs for the measurement harness (profiles/): variant and its two parameters
        if (const char* v = getenv("SVSB_GEMV_VARIANT")) { int x = atoi(v); if (x == 1 || x == 2) variant = x; }
        if (const char* v = getenv("SVSB_GEMV_TUNE_A")) tune_a = atoi(v);
        if (const char* v = getenv("SVSB_GEMV_TUNE_B")) tune_b = atoi(v);
    }
    if (variant == 2) {
        // tune_a = tile rows, tune_b = stages + 100 * consumer warps (e.g. 1604 = 16 warps, 4 stages)
        cudaError_t e = run_tma(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_a, tune_b % 100, tune_b / 100, reserve_sms);
        if (e != cudaErrorInvalidConfiguration) return e;
        (void)cudaGetLastError();
        tune_a = 0; tune_b = 0;                               // TMA knobs mean nothing to the LDG kernel
    }
    // LDG variant; tune_a selects the (R, U, THREADS) instantiation, tune_b caps blocks per SM
    switch (tune_a) {
        case 1:  return run_ldg<4, 2, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 2:  return run_ldg<4, 3, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 3:  return run_ldg<8, 1, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 4:  return run_ldg<8, 2, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 5:  return run_ldg<2, 4, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 6:  return run_ldg<2, 6, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 7:  return run_ldg<4, 3, 512>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 8:  return run_ldg<4, 4, 128>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        case 9:  return run_ldg<8, 3, 128>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
        default: return run_ldg<4, 3, 256>(st, device, M, n, d4, q, scores, gmax, group_shift, live, tune_b);
    }
}

cudaError_t launch_rows_to_i8(cudaStream_t st, int device, const float* M, int64_t n, int ld, void* M8, int ld8, float* scale8,
                              float* emax)
{
    if (n <= 0) return cudaSuccess;
    if (ld8 < ld || (ld8 & 15) || (ld & 3)) return cudaErrorInvalidValue;
    int64_t blocks = (n + 7) / 8;
    const int64_t cap = (int64_t)sm_count(device) * 16;
    if (blocks > cap) blocks = cap;
    rows_to_i8_kernel<<<(unsigned)blocks, 256, 0, st>>>(M, n, ld, static_cast<int8_t*>(M8), ld8, scale8, reinterpret_cast<uint32_t*>(emax));
    count_launch();
    return cudaGetLastError();
}

template <int CW, int NC>
static cudaError_t run_filter8_inst(cudaStream_t st, int64_t grid, size_t smem, const void* M8, const float* scale8, int64_t n, int c8,
                                    int tile_rows, int stages, const float* q, int ld, float* scores, u64* gmax, int group_shift,
                                    const uint8_t* live)
{
    auto kern = gemv8_tma_kernel<CW, NC>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = launch_kernel(kern, dim3((unsigned)grid), dim3((CW + 1) * 32), smem, st, static_cast<const int8_t*>(M8), scale8, n, c8,
                      tile_rows, stages, q, ld, scores, gmax, group_shift, live);
    count_launch();
    return e != cudaSuccess ? e : cudaGetLastError();
}

cudaError_t launch_filter8(cudaStream_t st, int device, const void* M8, const float* scale8, int64_t n, int ld, int ld8,
                           const float* q, float* scores, u64* gmax, int group_shift, int reserve_sms, const uint8_t* live)
{
    if (n <= 0) return cudaSuccess;
    if (ld > FILTER_MAX_LD || ld8 < ld || (ld8 & 15)) return cudaErrorInvalidValue;
    const int c8 = ld8 / 16;
    const size_t row_bytes = (size_t)ld8;
    // K1's ring: ~48 KB tiles x 3 stages (profiles/r01_tune_gemv.md)
    int tile_rows = 64;
    while (tile_rows > 1 && (size_t)tile_rows * row_bytes > 48 * 1024) tile_rows >>= 1;
    const int stages = 3;
    // the side data's bulk copies need 16-byte aligned sources: scale8 + r0 and live + r0 with r0 a multiple of tile_rows
    if (tile_rows % 16 || (reinterpret_cast<uintptr_t>(scale8) & 15) || (reinterpret_cast<uintptr_t>(live) & 15))
        return cudaErrorInvalidValue;
    const size_t smem = filter8_smem_bytes(tile_rows, stages, ld8);
    const int64_t ntiles = (n + tile_rows - 1) / tile_rows;
    int64_t grid = sm_count(device) - reserve_sms;
    if (grid > ntiles) grid = ntiles;
    if (grid < 1) grid = 1;
#define SVSB_F8_CASE(NCV) \
    return run_filter8_inst<8, NCV>(st, grid, smem, M8, scale8, n, c8, tile_rows, stages, q, ld, scores, gmax, group_shift, live)
    if (c8 <= 32) SVSB_F8_CASE(1);
    if (c8 <= 64) SVSB_F8_CASE(2);
    if (c8 <= 96) SVSB_F8_CASE(3);
    if (c8 <= 128) SVSB_F8_CASE(4);
    SVSB_F8_CASE(6);
#undef SVSB_F8_CASE
}

template <int NQ>
static cudaError_t run_rescore_inst(cudaStream_t st, int device, const float* M, int64_t n, int d4, const float* q, float* scores,
                                    u64* gmax, int group_shift, const uint8_t* live, uint32_t* state)
{
    const int64_t G = (n + ((int64_t)1 << group_shift) - 1) >> group_shift;
    int64_t blocks = (G + 7) / 8;
    const int64_t cap = (int64_t)sm_count(device) * 4;
    if (blocks > cap) blocks = cap;
    filter_rescore_kernel<NQ><<<(unsigned)blocks, 256, 0, st>>>(M, n, d4, q, scores, gmax, group_shift, live, state);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_filter_refine(cudaStream_t st, int device, const float* M, int64_t n, int ld, const float* q, float* scores,
                                 u64* gmax, int group_shift, int kk, float max_row_norm, const float* e8, const uint8_t* live,
                                 uint32_t* state)
{
    if (n <= 0) return cudaSuccess;
    if (ld > FILTER_MAX_LD) return cudaErrorInvalidValue;
    const int64_t G = (n + ((int64_t)1 << group_shift) - 1) >> group_shift;
    if (G > GROUPS_TARGET) return cudaErrorInvalidValue;
    filter_threshold_kernel<<<1, FT_THREADS, 0, st>>>(gmax, (int)G, kk, q, ld, max_row_norm, e8, state);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int d4 = ld / 4;
    if (d4 <= 64) return run_rescore_inst<2>(st, device, M, n, d4, q, scores, gmax, group_shift, live, state);
    if (d4 <= 192) return run_rescore_inst<6>(st, device, M, n, d4, q, scores, gmax, group_shift, live, state);
    if (d4 <= 384) return run_rescore_inst<12>(st, device, M, n, d4, q, scores, gmax, group_shift, live, state);
    return run_rescore_inst<24>(st, device, M, n, d4, q, scores, gmax, group_shift, live, state);
}

// ---- multi-query launcher ---------------------------------------------------------------------
template <int NQ, int BQ, bool FULL>
static cudaError_t run_mq_inst2(cudaStream_t st, int64_t grid, size_t smem, const float* M, int64_t n, int d4, int tile_rows, int stages,
                               const float* Q, int b, int groups, float* scores, int64_t n_stride, u64* gmax, int64_t g_stride,
                               int group_shift, const uint8_t* live)
{
    auto kern = gemv_tma_mq_kernel<NQ, BQ, FULL>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)grid, 384, smem, st>>>(M, n, d4, tile_rows, stages, Q, b, groups, scores, n_stride, gmax, g_stride, group_shift, live);
    count_launch();
    return cudaGetLastError();
}

template <int NQ, int BQ>
static cudaError_t run_mq_inst(cudaStream_t st, int64_t grid, size_t smem, const float* M, int64_t n, int d4, int tile_rows, int stages,
                               const float* Q, int b, int groups, float* scores, int64_t n_stride, u64* gmax, int64_t g_stride,
                               int group_shift, const uint8_t* live)
{
    if (d4 == 32 * NQ)
        return run_mq_inst2<NQ, BQ, true>(st, grid, smem, M, n, d4, tile_rows, stages, Q, b, groups, scores, n_stride, gmax, g_stride, group_shift, live);
    return run_mq_inst2<NQ, BQ, false>(st, grid, smem, M, n, d4, tile_rows, stages, Q, b, groups, scores, n_stride, gmax, g_stride, group_shift, live);
}

int gemv_mq_queries_per_warp(int ld) {
    const int d4 = ld / 4;
    return d4 <= 64 ? 8 : d4 <= 192 ? 4 : d4 <= 384 ? 4 : d4 <= 768 ? 2 : 0;   // 16 * NQ * BQ query + 8 * BQ accumulator registers <= ~224
}

cudaError_t launch_gemv_mq(cudaStream_t st, int device, const float* M, int64_t n, int d, int ld, const float* Q, int b,
                           float* scores, int64_t n_stride, u64* gmax, int64_t g_stride, int group_shift, const uint8_t* live,
                           int reserve_sms)
{
    (void)d;
    if (n <= 0 || b <= 0) return cudaSuccess;
    const int d4 = ld / 4;
    const int bq_hi = gemv_mq_queries_per_warp(ld);
    if (bq_hi == 0) return cudaErrorInvalidConfiguration;       // rows too long for register-resident queries
    int bq = bq_hi;
    if (bq_hi > 2 && b <= bq_hi / 2) bq = bq_hi / 2;             // fewer wasted FMAs for a small batch
    int groups = 1;
    while (groups * bq < b) groups <<= 1;
    if (groups > 8) return cudaErrorInvalidConfiguration;       // the caller chunks larger batches
    const size_t row_bytes = (size_t)d4 * 16;
    int tile_rows = 64;
    while (tile_rows > 1 && (size_t)tile_rows * row_bytes > 48 * 1024) tile_rows >>= 1;
    if (tile_rows < 8 / groups) { /* every warp of a group still gets whole rows: fine, some idle */ }
    const int stages = 3;
    const size_t smem = (size_t)stages * tile_rows * row_bytes + (size_t)stages * 16 + 64;
    const int64_t ntiles = (n + tile_rows - 1) / tile_rows;
    int64_t grid = sm_count(device) - reserve_sms;
    if (grid > ntiles) grid = ntiles;
    if (grid < 1) grid = 1;
    const int nq = d4 <= 64 ? 2 : d4 <= 192 ? 6 : d4 <= 384 ? 12 : 24;
#define SVSB_MQ_CASE(NQV, BQV) \
    return run_mq_inst<NQV, BQV>(st, grid, smem, M, n, d4, tile_rows, stages, Q, b, groups, scores, n_stride, gmax, g_stride, group_shift, live)
    switch (nq * 100 + bq) {
        case 204: SVSB_MQ_CASE(2, 4);
        case 208: SVSB_MQ_CASE(2, 8);
        case 602: SVSB_MQ_CASE(6, 2);
        case 604: SVSB_MQ_CASE(6, 4);
        case 1202: SVSB_MQ_CASE(12, 2);
        case 1204: SVSB_MQ_CASE(12, 4);
        case 2402: SVSB_MQ_CASE(24, 2);
        default: return cudaErrorInvalidConfiguration;
    }
#undef SVSB_MQ_CASE
}

}  // namespace svsb
