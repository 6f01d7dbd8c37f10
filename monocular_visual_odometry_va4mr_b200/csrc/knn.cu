// Brute-force kNN(k=2) + Lowe ratio test for SIFT descriptors (replaces
// cv2.BFMatcher().knnMatch(d0, d1, k=2) at reference VisualOdometryPipeLine.py:229 and the Python
// ratio loop at :218-224; spec SURVEY.md A.5).
//
// d^2(i,j) = |q_i|^2 + |t_j|^2 - 2 q_i.t_j.  OpenCV's SIFT descriptors are integers 0..255, so fp16
// operands with fp32 accumulation give the dot products exactly (every partial sum is an integer
// < 2^24) and the squared distances are exact integers: indices, tie-breaks (lowest train index
// first) and the ratio decision are bit-exact with cv2.
//
// The contraction runs on the 5th-gen tensor cores: tcgen05.mma (cta_group::1, kind::f16,
// M=128, N=128, K=16 x 9) issued by one thread, operands staged by TMA into swizzled shared
// memory, accumulators double-buffered in TMEM (2 stages x 2 query halves x 128 columns).  Sixteen
// epilogue warps (four per TMEM lane quadrant) pull the accumulators with tcgen05.ld and keep a running
// (best, second) per query row in registers -- the Q x T distance matrix is never materialised.  A CTA
// owns a contiguous run of (query pair, train tile) units; partial top-2s of the runs are merged in
// index order.
#include "internal.cuh"
#include "tma.cuh"
#include <cuda_fp16.h>

#define KNN_BM 128
#define KNN_DIM 128
#define KNN_EPI_WARPS 16
#define KNN_THREADS (64 + 32 * KNN_EPI_WARPS)
#define KNN_BIG 3.0e38f

// ------------------------------------------------------------------ PTX wrappers (TMA/mbarrier: tma.cuh)
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// K-major, 128B-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr)
{
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

struct KnnPartial { float d1, d2; int i1, i2; };

// ------------------------------------------------------------------ GEMM + fused top-2: 256 query rows per CTA, distances inside the GEMM
// At 8192 x 8192 two things bound a tensor-core kNN (DESIGN.md section 4): the L2 operand feed -- every CTA streams the
// train descriptors -- and the scan, where a compare-select update path is entered by a warp whenever ANY of its 32 rows
// is displaced, i.e. for about half of the four-column groups.  This kernel
//  (1) keeps TWO query tiles resident per CTA and streams train tiles of 128 rows through a 3-stage ring, so one 36 KB
//      stage feeds two M = 128 MMAs (half the operand bytes per flop of a single query tile);
//  (2) lets the tensor core produce the finished squared distance, offset into one binade: seven extra K columns carry
//      |t|^2 and |q|^2 as base-256 digits against {1, 256, 256} and the constant 2^23 = 4096 * 2048, so the accumulator
//      is  d + 2^23  with d = |q|^2 + |t|^2 - 2 q.t in [0, 128 * 255^2] -- an integer in [2^23, 2^24), whose float32 bit
//      pattern is 0x4B000000 | d.  Every operand is an integer fp16 holds exactly and every partial sum an integer below
//      2^24, so this is exact.  The 16 extra K columns travel as their own 32-byte-swizzled TMA boxes and cost one more
//      UMMA_K step (K = 144);
//  (3) scans WITHOUT a branch: key = bits * 64 + (0x80000000 | column) = 0x40000000 | d << 6 | column is a positive normal
//      float pattern ordered like (d, column), so a min / max network of FMNMX / FMNMX3 on the keys gives the two smallest
//      (distance, lowest column first) of the thread's 64 columns in ~220 independent instructions -- no update path, no
//      shared bounds, no dependence on the data;
//  (4) spreads (query pair, train tile) units over all SMs in contiguous runs (a run may cross into the next query pair:
//      the A tiles are reloaded and the rows' partial top-2 go to the CTA's slot of that pair).
#define K3_BN 128
#define K3_STAGES 3
#define K3_A_HALF (KNN_BM * KNN_DIM * 2 + KNN_BM * 32)        // 32 KB main + 4 KB extra columns
#define K3_B_STAGE (K3_BN * KNN_DIM * 2 + K3_BN * 32)         // 32 KB + 4 KB
#define K3_SMEM (1024 + 2 * K3_A_HALF + K3_STAGES * K3_B_STAGE + 256)

__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr)
{
    // K-major, 32-byte swizzle: rows of 32 B, 8-row groups 256 B apart
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | (16ull << 32) | (1ull << 46) | (6ull << 61);
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t* v)
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld_wait16(uint32_t* v)
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :: "memory");
}
__device__ __forceinline__ float fmin3(float a, float b, float c)
{
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// f32 -> fp16 operands of the kernel below.  Extra K columns (16 per row):
//   query: -2 q | {1, 256, 256,  q0, q1, 256 q2,  4096, 0 ..}     train: t | {a0, a1, 256 a2,  1, 256, 256,  2048, 0 ..}
// with |q|^2 = q0 + 256 q1 + 65536 q2 and |t|^2 = a0 + 256 a1 + 65536 a2: the extra columns contribute
// |t|^2 + |q|^2 + 2^23.  Rows beyond n are zero vectors (their columns are masked in the scan / dropped in the merge).
__global__ void __launch_bounds__(256)
knn_prep3_kernel(const float* __restrict__ src, int n, int n_pad, int is_query, __half* __restrict__ dst, __half* __restrict__ ext,
                 float* __restrict__ norm, int* __restrict__ bad)
{
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n_pad) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < n) v = reinterpret_cast<const float4*>(src + (size_t)row * KNN_DIM)[lane];
    const float a[4] = {v.x, v.y, v.z, v.w};
    float s = 0.f;
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        ok = ok && (a[k] >= 0.f) && (a[k] <= 255.f) && (a[k] == floorf(a[k]));
        s += a[k] * a[k];
    }
    const float sc = is_query ? -2.f : 1.f;
    __half2 h0 = __floats2half2_rn(sc * a[0], sc * a[1]), h1 = __floats2half2_rn(sc * a[2], sc * a[3]);
    uint2 pk;
    pk.x = *reinterpret_cast<uint32_t*>(&h0);
    pk.y = *reinterpret_cast<uint32_t*>(&h1);
    reinterpret_cast<uint2*>(dst + (size_t)row * KNN_DIM)[lane] = pk;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);   // exact: integers < 2^24
    if (!__all_sync(0xffffffffu, ok) && lane == 0) atomicOr(bad, 1);
    if (lane == 0 && norm) norm[row] = s;
    if (lane < 16) {
        const int si = (ok && row < n) ? (int)s : 0;
        const float dig = lane % 3 == 0 ? (float)(si & 255) : lane % 3 == 1 ? (float)((si >> 8) & 255) : (float)((si >> 16) * 256);
        const float one = lane % 3 == 0 ? 1.f : 256.f;
        float e = 0.f;
        if (lane < 3) e = is_query ? one : dig;          // against the train row's |t|^2 digits
        else if (lane < 6) e = is_query ? dig : one;     // the query row's |q|^2 digits
        else if (lane == 6) e = is_query ? 4096.f : 2048.f;
        ext[(size_t)row * 16 + lane] = __float2half_rn(e);
    }
}

__global__ void __launch_bounds__(KNN_THREADS, 1)
knn_gemm_top2_m256_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_qx,
                          const __grid_constant__ CUtensorMap map_t, const __grid_constant__ CUtensorMap map_tx,
                          int n_tiles, int per, int total, int nt, KnnPartial* __restrict__ partial, int nq_pad)
{
    extern __shared__ uint8_t smem_raw[];
    const int f0 = blockIdx.x * per, f1 = min(f0 + per, total);
    if (f0 >= f1) return;                      // uniform: before any barrier / TMEM allocation
    const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t sA = base;
    const uint32_t sB = base + 2 * K3_A_HALF;
    const uint32_t sBar = sB + K3_STAGES * K3_B_STAGE;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem_raw + (sBar + 128 - smem_u32(smem_raw)));
    // accumulator barriers per (TMEM stage, query half): the eight epilogue warps of a half start on its 128 columns while
    // the MMAs of the other half are still running
    const uint32_t bar_a = sBar, bar_aempty = sBar + 8, bar_bfull = sBar + 16, bar_bempty = sBar + 40, bar_accfull = sBar + 64,
                   bar_accempty = sBar + 96;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        mbar_init(bar_a, 1);
        mbar_init(bar_aempty, 1);
        for (int s = 0; s < K3_STAGES; ++s) { mbar_init(bar_bfull + 8 * s, 1); mbar_init(bar_bempty + 8 * s, 1); }
        for (int s = 0; s < 4; ++s) { mbar_init(bar_accfull + 8 * s, 1); mbar_init(bar_accempty + 8 * s, 32 * KNN_EPI_WARPS / 2); }
        mbar_fence_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int it = 0, seg = 0;
            for (int f = f0; f < f1; ++seg) {
                const int m = f / n_tiles, na = f - m * n_tiles, nb = min(n_tiles, na + (f1 - f));
                mbar_wait(bar_aempty, (seg & 1) ^ 1);            // the previous segment's MMAs have read the old A tiles
                mbar_expect_tx(bar_a, 2 * K3_A_HALF);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t dst = sA + h * K3_A_HALF;
                    const int r0 = m * 2 * KNN_BM + h * KNN_BM;
                    tma_load_2d(dst, &map_q, 0, r0, bar_a);
                    tma_load_2d(dst + KNN_BM * 128, &map_q, 64, r0, bar_a);
                    tma_load_2d(dst + KNN_BM * 256, &map_qx, 0, r0, bar_a);
                }
                for (int n = na; n < nb; ++n, ++it) {
                    const int s = it % K3_STAGES, ph = (it / K3_STAGES) & 1;
                    mbar_wait(bar_bempty + 8 * s, ph ^ 1);
                    mbar_expect_tx(bar_bfull + 8 * s, K3_B_STAGE);
                    const uint32_t dst = sB + s * K3_B_STAGE;
                    tma_load_2d(dst, &map_t, 0, n * K3_BN, bar_bfull + 8 * s);
                    tma_load_2d(dst + K3_BN * 128, &map_t, 64, n * K3_BN, bar_bfull + 8 * s);
                    tma_load_2d(dst + K3_BN * 256, &map_tx, 0, n * K3_BN, bar_bfull + 8 * s);
                }
                f += nb - na;
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // instruction descriptor: D=F32, A=B=F16, K-major both, N=128, M=128
            const uint32_t idesc = (1u << 4) | ((uint32_t)(K3_BN >> 3) << 17) | ((uint32_t)(KNN_BM >> 4) << 24);
            int it = 0, seg = 0;
            for (int f = f0; f < f1; ++seg) {
                const int m = f / n_tiles, na = f - m * n_tiles, nb = min(n_tiles, na + (f1 - f));
                mbar_wait(bar_a, seg & 1);
                for (int n = na; n < nb; ++n, ++it) {
                    const int s = it % K3_STAGES, ph = (it / K3_STAGES) & 1;
                    const int as = it & 1, aph = (it >> 1) & 1;
                    mbar_wait(bar_bfull + 8 * s, ph);
                    const uint32_t sBs = sB + s * K3_B_STAGE;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        mbar_wait(bar_accempty + 8 * (as * 2 + h), aph ^ 1);
                        tc_fence_after();
                        const uint32_t d_tmem = tmem_base + (uint32_t)(as * 256 + h * 128);
                        const uint32_t sAh = sA + h * K3_A_HALF;
#pragma unroll
                        for (int kb = 0; kb < 2; ++kb) {
                            const uint64_t adesc = umma_desc_sw128(sAh + kb * (KNN_BM * 128));
                            const uint64_t bdesc = umma_desc_sw128(sBs + kb * (K3_BN * 128));
#pragma unroll
                            for (int k = 0; k < 4; ++k)   // 16 fp16 = 32 B per UMMA_K step inside the swizzle atom
                                tc_mma_f16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
                        }
                        tc_mma_f16(d_tmem, umma_desc_sw32(sAh + KNN_BM * 256), umma_desc_sw32(sBs + K3_BN * 256), idesc, 1);   // the norm columns
                        if (h == 1) tc_commit(bar_bempty + 8 * s);              // smem stage free once these MMAs have read it
                        tc_commit(bar_accfull + 8 * (as * 2 + h));              // this half's accumulator is ready for the epilogue
                    }
                }
                tc_commit(bar_aempty);                  // every MMA of this segment has read the A tiles
                f += nb - na;
            }
        }
    } else {
        // epilogue: warp w may touch TMEM lanes 32*(w%4) .. +31.  Sixteen warps = 4 lane quadrants x 2 query halves x 2
        // column groups of 64; one query row per thread.  The accumulator holds d + 2^23 (see above).
        const int q = warp & 3;
        const int idx = (warp - 2) >> 2;
        const int h = idx >> 1, cg = idx & 1;
        const int rl = h * KNN_BM + q * 32 + lane;          // row inside the query pair
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * 128 + cg * 64);
        const int pad_tile = (nt % K3_BN) ? n_tiles - 1 : -1;   // the train tile that holds rows beyond nt
        int it = 0;
        uint32_t va[16], vb[16];
        {   // first 16-column piece of the first unit; from here on the pieces form one software pipeline across units and
            // segments: while a piece is reduced the next one's tcgen05.ld is in flight
            mbar_wait(bar_accfull + 8 * h, 0);
            tc_fence_after();
            tc_ld16(lane_base, va);
        }
        for (int f = f0; f < f1;) {
            const int m = f / n_tiles, na = f - m * n_tiles, nb = min(n_tiles, na + (f1 - f));
            const int row = m * 2 * KNN_BM + rl;
            // running two smallest of this row over the segment's train tiles: (distance, train index), earlier tiles win ties
            int r1d = 0x7FFFFFFF, r2d = 0x7FFFFFFF, r1i = -1, r2i = -1;
            for (int n = na; n < nb; ++n, ++it) {
                const int as = it & 1;
                const int j0 = n * K3_BN + cg * 64;
                float s1[4], s2[4];     // the two smallest keys of each 16-column piece
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    uint32_t* v = (c & 1) ? vb : va;
                    tc_ld_wait16(v);
                    if (c < 3) {
                        tc_ld16(lane_base + (uint32_t)(as * 256 + (c + 1) * 16), (c & 1) ? va : vb);   // in flight while this piece is reduced
                    } else {
                        tc_fence_before();
                        mbar_arrive(bar_accempty + 8 * (as * 2 + h));                 // all four pieces are in registers
                    }
                    // key = bits * 64 + (0x80000000 | column) = 0x40000000 | d << 6 | column: positive normal float patterns
                    // ordered like (d, column)
                    float k[16];
#pragma unroll
                    for (int e = 0; e < 16; ++e) k[e] = __uint_as_float(v[e] * 64u + (0x80000000u | (uint32_t)(c * 16 + e)));
                    if (c == 3 && f + (n - na) + 1 < f1) {                            // first piece of the next unit (vb's keys are built, va is free)
                        const int it2 = it + 1;
                        mbar_wait(bar_accfull + 8 * ((it2 & 1) * 2 + h), (it2 >> 1) & 1);
                        tc_fence_after();
                        tc_ld16(lane_base + (uint32_t)((it2 & 1) * 256), va);
                    }
                    if (n == pad_tile) {      // rows beyond nt: never candidates
#pragma unroll
                        for (int e = 0; e < 16; ++e) k[e] = (j0 + c * 16 + e) < nt ? k[e] : __uint_as_float(0x7F000000u);
                    }
                    // two smallest of 16 distinct keys: sorted pairs, then merges (a1 <= a2) + (b1 <= b2) ->
                    // (min(a1, b1), min(max(a1, b1), a2, b2))
                    float lo[8], hi[8];
#pragma unroll
                    for (int e = 0; e < 8; ++e) { lo[e] = fminf(k[2 * e], k[2 * e + 1]); hi[e] = fmaxf(k[2 * e], k[2 * e + 1]); }
#pragma unroll
                    for (int w = 4; w >= 1; w >>= 1) {
#pragma unroll
                        for (int e = 0; e < w; ++e) {
                            const float a1 = lo[e], b1 = lo[e + w];
                            lo[e] = fminf(a1, b1);
                            hi[e] = fmin3(fmaxf(a1, b1), hi[e], hi[e + w]);
                        }
                    }
                    s1[c] = lo[0]; s2[c] = hi[0];
                }
                // the four pieces' pairs -> the stage's two smallest (keys order ties by column)
#pragma unroll
                for (int w = 2; w >= 1; w >>= 1) {
#pragma unroll
                    for (int e = 0; e < w; ++e) {
                        const float a1 = s1[e], b1 = s1[e + w];
                        s1[e] = fminf(a1, b1);
                        s2[e] = fmin3(fmaxf(a1, b1), s2[e], s2[e + w]);
                    }
                }
                const float t1 = s1[0], t2 = s2[0];
                const uint32_t u1 = __float_as_uint(t1), u2 = __float_as_uint(t2);
                const int n1d = (int)((u1 >> 6) & 0x7FFFFFu), n2d = (int)((u2 >> 6) & 0x7FFFFFu);
                const int n1i = u1 >= 0x7F000000u ? -1 : j0 + (int)(u1 & 63u), n2i = u2 >= 0x7F000000u ? -1 : j0 + (int)(u2 & 63u);
                const int m1d = n1i < 0 ? 0x7FFFFFFF : n1d, m2d = n2i < 0 ? 0x7FFFFFFF : n2d;
                // merge into the running pair; on equal distance the running entry (a lower train index) stays ahead
                const bool first = m1d < r1d;
                const int o2d = first ? (r1d <= m2d ? r1d : m2d) : (m1d < r2d ? m1d : r2d);
                const int o2i = first ? (r1d <= m2d ? r1i : n2i) : (m1d < r2d ? n1i : r2i);
                r1i = first ? n1i : r1i;
                r1d = first ? m1d : r1d;
                r2d = o2d; r2i = o2i;
            }
            KnnPartial p;
            p.d1 = r1i >= 0 ? (float)r1d : KNN_BIG;
            p.d2 = r2i >= 0 ? (float)r2d : KNN_BIG;
            p.i1 = r1i; p.i2 = r2i;
            const int slot = (int)blockIdx.x - (m * n_tiles) / per;       // this CTA's position among those sharing query pair m
            partial[((size_t)slot * 2 + cg) * nq_pad + row] = p;
            f += nb - na;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// merge the per-range partial top-2s in train-index order, take square roots, apply the ratio test
__global__ void __launch_bounds__(256)
knn_finalize_kernel(const KnnPartial* __restrict__ partial, int n_lists, int nq, int nq_pad, int nt, double ratio,
                    int* __restrict__ idx2, float* __restrict__ dist2, uint8_t* __restrict__ accept)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nq) return;
    float b1 = KNN_BIG, b2 = KNN_BIG;
    int i1 = -1, i2 = -1;
    for (int s = 0; s < n_lists; ++s) {
        const KnnPartial p = partial[(size_t)s * nq_pad + r];
        const float ds[2] = {p.d1, p.d2};
        const int is[2] = {p.i1, p.i2};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float d = ds[k];
            const int j = is[k];
            if (j < 0 || j >= nt) continue;
            // partial lists interleave in train index: order by (distance, index)
            const bool lt1 = d < b1 || (d == b1 && j < i1), lt2 = d < b2 || (d == b2 && j < i2);
            i2 = lt1 ? i1 : (lt2 ? j : i2);
            b2 = lt1 ? b1 : (lt2 ? d : b2);
            i1 = lt1 ? j : i1;
            b1 = lt1 ? d : b1;
        }
    }
    const float FMAX = 3.402823466e+38f;
    const float d1 = i1 >= 0 ? __fsqrt_rn(b1) : FMAX;
    const float d2 = i2 >= 0 ? __fsqrt_rn(b2) : FMAX;
    idx2[2 * r] = i1; idx2[2 * r + 1] = i2;
    dist2[2 * r] = d1; dist2[2 * r + 1] = d2;
    // reference :221  m.distance < feature_ratio * n.distance, evaluated in Python float64
    accept[r] = (i1 >= 0 && i2 >= 0 && (double)d1 < __dmul_rn(ratio, (double)d2)) ? 1 : 0;
}

// ------------------------------------------------------------------ host
static int knn_make_map(b200vo_ctx* ctx, CUtensorMap* map, void* gptr, int rows, int box_rows)
{
    const cuuint64_t dims[2] = {(cuuint64_t)KNN_DIM, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)KNN_DIM * 2};
    const cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    return vo_encode_tiled(ctx, map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, gptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B);
}

static int knn_make_map_ext(b200vo_ctx* ctx, CUtensorMap* map, void* gptr, int rows, int box_rows)
{
    const cuuint64_t dims[2] = {16, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {32};
    const cuuint32_t box[2] = {16, (cuuint32_t)box_rows};
    return vo_encode_tiled(ctx, map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, gptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}

// scratch of vo_knn2_ratio_dev for nq queries and nt train descriptors (bytes of ctx->d_scratch[3])
size_t vo_knn2_workspace(const b200vo_ctx* ctx, int nq, int nt)
{
    const int nq_pad = (int)vo_align((size_t)nq, 2 * KNN_BM), nt_pad = (int)vo_align((size_t)nt, K3_BN);
    const int m_pairs = nq_pad / (2 * KNN_BM), n_tiles = nt_pad / K3_BN;
    const int total = m_pairs * n_tiles;
    const int per = (total + ctx->num_sms - 1) / ctx->num_sms;
    const int n_splits = (n_tiles + per - 1) / per + 1;
    const size_t b_q16 = vo_align((size_t)nq_pad * KNN_DIM * 2, 1024), b_t16 = vo_align((size_t)nt_pad * KNN_DIM * 2, 1024);
    const size_t b_qx = vo_align((size_t)nq_pad * 32, 1024), b_tx = vo_align((size_t)nt_pad * 32, 1024);
    const size_t b_part = vo_align((size_t)2 * n_splits * nq_pad * sizeof(KnnPartial), 256);
    return b_q16 + b_t16 + b_qx + b_tx + b_part + 256;
}

// device-resident core: q_dev/t_dev float32 row-major; outputs device pointers
int vo_knn2_ratio_dev(b200vo_ctx* ctx, const float* q_dev, int nq, const float* t_dev, int nt, double ratio,
                      int* idx2_dev, float* dist2_dev, uint8_t* accept_dev, int* bad_flag_host)
{
    const int nq_pad = (int)vo_align((size_t)nq, 2 * KNN_BM), nt_pad = (int)vo_align((size_t)nt, K3_BN);
    const int m_pairs = nq_pad / (2 * KNN_BM), n_tiles = nt_pad / K3_BN;
    // (query pair, train tile) units in query-pair-major order, one contiguous run per SM
    const int total = m_pairs * n_tiles;
    const int per = (total + ctx->num_sms - 1) / ctx->num_sms;
    const int n_splits = (n_tiles + per - 1) / per + 1;      // CTAs that can share one query pair
    const size_t b_q16 = vo_align((size_t)nq_pad * KNN_DIM * 2, 1024), b_t16 = vo_align((size_t)nt_pad * KNN_DIM * 2, 1024);
    const size_t b_qx = vo_align((size_t)nq_pad * 32, 1024), b_tx = vo_align((size_t)nt_pad * 32, 1024);
    const size_t b_part = vo_align((size_t)2 * n_splits * nq_pad * sizeof(KnnPartial), 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[3], vo_knn2_workspace(ctx, nq, nt)));
    uint8_t* d = (uint8_t*)ctx->d_scratch[3].p;
    __half* q16 = (__half*)d; d += b_q16;
    __half* t16 = (__half*)d; d += b_t16;
    __half* qx = (__half*)d; d += b_qx;
    __half* tx = (__half*)d; d += b_tx;
    KnnPartial* part = (KnnPartial*)d; d += b_part;
    int* bad = (int*)d;
    ctx->knn_bad_flag = bad;
    VO_CUDA(ctx, cudaMemsetAsync(bad, 0, 4, ctx->stream));
    VO_CUDA(ctx, cudaMemsetAsync(part, 0xFF, b_part, ctx->stream));   // lists no CTA writes: index -1 = "no entry"
    knn_prep3_kernel<<<(nq_pad + 7) / 8, 256, 0, ctx->stream>>>(q_dev, nq, nq_pad, 1, q16, qx, nullptr, bad);
    knn_prep3_kernel<<<(nt_pad + 7) / 8, 256, 0, ctx->stream>>>(t_dev, nt, nt_pad, 0, t16, tx, nullptr, bad);
    ctx->launches += 2;
    CUtensorMap map_q, map_t, map_qx, map_tx;
    VO_TRY(knn_make_map(ctx, &map_q, q16, nq_pad, KNN_BM));
    VO_TRY(knn_make_map(ctx, &map_t, t16, nt_pad, K3_BN));
    VO_TRY(knn_make_map_ext(ctx, &map_qx, qx, nq_pad, KNN_BM));
    VO_TRY(knn_make_map_ext(ctx, &map_tx, tx, nt_pad, K3_BN));
    static bool attr_done = false;
    if (!attr_done) {
        VO_CUDA(ctx, cudaFuncSetAttribute(knn_gemm_top2_m256_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, K3_SMEM));
        attr_done = true;
    }
    knn_gemm_top2_m256_kernel<<<(total + per - 1) / per, KNN_THREADS, K3_SMEM, ctx->stream>>>(map_q, map_qx, map_t, map_tx, n_tiles, per, total, nt,
                                                                                               part, nq_pad);
    knn_finalize_kernel<<<(nq + 255) / 256, 256, 0, ctx->stream>>>(part, 2 * n_splits, nq, nq_pad, nt, ratio, idx2_dev, dist2_dev, accept_dev);
    ctx->launches += 2;
    VO_CUDA(ctx, cudaGetLastError());
    if (bad_flag_host) VO_CUDA(ctx, cudaMemcpyAsync(bad_flag_host, bad, 4, cudaMemcpyDeviceToHost, ctx->stream));
    return 0;
}

// Device-pointer form (SURVEY 8b `_dev`): descriptors already in device memory, results left there; asynchronous on
// the ctx stream.  bad_dev (may be NULL) int32[1]: 1 when a descriptor is not integer-valued in 0..255.
__global__ void knn_export_flag_kernel(const int* __restrict__ bad, int32_t* __restrict__ out) { *out = *bad ? 1 : 0; }
__global__ void knn_empty_train_kernel(int nq, int32_t* __restrict__ idx2, float* __restrict__ dist2, uint8_t* __restrict__ accept)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    idx2[2 * i] = idx2[2 * i + 1] = -1;
    dist2[2 * i] = dist2[2 * i + 1] = 3.402823466e+38f;
    accept[i] = 0;
}

extern "C" int b200vo_knn2_ratio_dev(b200vo_ctx* ctx, const float* q_dev, int nq, const float* t_dev, int nt, int dim, double ratio,
                                     int32_t* idx2_dev, float* dist2_dev, uint8_t* accept_dev, int32_t* bad_dev)
{
    if (!ctx || !q_dev || !t_dev || !idx2_dev || !dist2_dev || !accept_dev) return B200VO_E_BADARG;
    if (nq < 0 || nt < 0 || dim <= 0) return vo_set_err(ctx, B200VO_E_BADARG, "type == src2.type() && src1.cols == src2.cols");
    if (dim != KNN_DIM) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "descriptor length %d != 128 (SIFT)", dim);
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    if (bad_dev) VO_CUDA(ctx, cudaMemsetAsync(bad_dev, 0, 4, ctx->stream));
    if (nq == 0) return 0;
    if (nt == 0) {
        knn_empty_train_kernel<<<(nq + 255) / 256, 256, 0, ctx->stream>>>(nq, idx2_dev, dist2_dev, accept_dev);
        ctx->launches++;
        return 0;
    }
    VO_TRY(vo_knn2_ratio_dev(ctx, q_dev, nq, t_dev, nt, ratio, idx2_dev, dist2_dev, accept_dev, nullptr));
    if (bad_dev) {
        // the flag vo_knn2_ratio_dev keeps at the end of its scratch block (see its carve-up)
        knn_export_flag_kernel<<<1, 1, 0, ctx->stream>>>(ctx->knn_bad_flag, bad_dev);
        ctx->launches++;
    }
    return 0;
}

extern "C" int b200vo_knn2_ratio(b200vo_ctx* ctx, const float* q, int nq, const float* t, int nt, int dim,
                                 double ratio, int32_t* idx2, float* dist2, uint8_t* accept)
{
    if (!ctx || !q || !t || !idx2 || !dist2 || !accept) return B200VO_E_BADARG;
    if (nq < 0 || nt < 0 || dim <= 0) return vo_set_err(ctx, B200VO_E_BADARG, "type == src2.type() && src1.cols == src2.cols");
    if (dim != KNN_DIM) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "descriptor length %d != 128 (SIFT)", dim);
    if (nq == 0) return 0;
    if (nt == 0) {
        for (int i = 0; i < nq; ++i) { idx2[2 * i] = idx2[2 * i + 1] = -1; dist2[2 * i] = dist2[2 * i + 1] = 3.402823466e+38f; accept[i] = 0; }
        return 0;
    }
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const size_t b_q = vo_align((size_t)nq * dim * 4, 256), b_t = vo_align((size_t)nt * dim * 4, 256);
    const size_t b_i = vo_align((size_t)nq * 8, 256), b_d = vo_align((size_t)nq * 8, 256), b_a = vo_align((size_t)nq, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[4], b_q + b_t + b_i + b_d + b_a));
    VO_TRY(vo_reserve_pinned(ctx, b_q + b_t + b_i + b_d + b_a + 256));
    uint8_t* dv = (uint8_t*)ctx->d_scratch[4].p;
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    // page-locked caller arrays (b200vo_host_alloc / cudaHostRegister) are DMA'd in place; pageable ones are staged
    auto is_pinned = [](const void* p) {
        cudaPointerAttributes a{};
        const bool r = cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost;
        cudaGetLastError();
        return r;
    };
    const void* qsrc = q;
    const void* tsrc = t;
    if (!is_pinned(q)) { memcpy(hp, q, (size_t)nq * dim * 4); qsrc = hp; }
    VO_CUDA(ctx, cudaMemcpyAsync(dv, qsrc, (size_t)nq * dim * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (!is_pinned(t)) { memcpy(hp + b_q, t, (size_t)nt * dim * 4); tsrc = hp + b_q; }
    VO_CUDA(ctx, cudaMemcpyAsync(dv + b_q, tsrc, (size_t)nt * dim * 4, cudaMemcpyHostToDevice, ctx->stream));
    int* h_bad = (int*)(hp + b_q + b_t + b_i + b_d + b_a);
    *h_bad = 0;
    VO_TRY(vo_knn2_ratio_dev(ctx, (const float*)dv, nq, (const float*)(dv + b_q), nt, ratio, (int*)(dv + b_q + b_t),
                             (float*)(dv + b_q + b_t + b_i), dv + b_q + b_t + b_i + b_d, h_bad));
    const bool o_pin = is_pinned(idx2) && is_pinned(dist2) && is_pinned(accept);
    if (o_pin) {
        VO_CUDA(ctx, cudaMemcpyAsync(idx2, dv + b_q + b_t, (size_t)nq * 8, cudaMemcpyDeviceToHost, ctx->stream));
        VO_CUDA(ctx, cudaMemcpyAsync(dist2, dv + b_q + b_t + b_i, (size_t)nq * 8, cudaMemcpyDeviceToHost, ctx->stream));
        VO_CUDA(ctx, cudaMemcpyAsync(accept, dv + b_q + b_t + b_i + b_d, (size_t)nq, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
        VO_CUDA(ctx, cudaMemcpyAsync(hp + b_q + b_t, dv + b_q + b_t, b_i + b_d + b_a, cudaMemcpyDeviceToHost, ctx->stream));
    }
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    if (*h_bad)
        return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "descriptors must be integer-valued in 0..255 (cv2 SIFT); other float descriptors are not implemented");
    if (!o_pin) {
        memcpy(idx2, hp + b_q + b_t, (size_t)nq * 8);
        memcpy(dist2, hp + b_q + b_t + b_i, (size_t)nq * 8);
        memcpy(accept, hp + b_q + b_t + b_i + b_d, (size_t)nq);
    }
    return 0;
}
