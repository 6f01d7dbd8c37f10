// Shi-Tomasi corner detection (replaces cv2.goodFeaturesToTrack at reference
// VisualOdometryPipeLine.py:256; spec SURVEY.md A.4 and the arithmetic pinned in
// oracle/gftt_oracle.c).
//
// The float32 operation order reproduces cv2 4.13's min-eigenvalue map bit for bit (fused
// multiply-adds exactly where its AVX2 filters fuse, box sums as a running column sum in
// double), because the ordered corner list is decided by last-bit ties between symmetric
// corners.  Pipeline:
//   gftt_cov_kernel        Sobel (scaled) -> Dx^2, DxDy, Dy^2             (1 thread / pixel)
//   gftt_rowsum/colsum/eig 3x3 box as running column sums in double (serial chain per column and plane), eig
//   gftt_candidates_kernel threshold at q*max, 3x3 non-maximum test, compaction of 64-bit keys
//   gftt_rank_kernel       order by (value desc, address desc): rank by counting (n <= 32768)
//   gftt_bitonic_*         same order for larger candidate sets
//   gftt_select_kernel     greedy min-distance suppression on a cell grid, warp-speculative:
//                          32 candidates tested against the accepted set at once, survivors
//                          resolved in order -- result identical to the sequential loop.
#include "internal.cuh"

__device__ __forceinline__ int refl101(int p, int len)
{
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

// img: bordered level-0 (REFLECT_101 border materialised), base -> pixel (0,0)
__global__ void __launch_bounds__(256)
gftt_cov_kernel(const uint8_t* __restrict__ img, size_t img_stride, int pitch, int w, int h, float k0, float k1,
                float* __restrict__ cov)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    img += blockIdx.z * img_stride;                       // one image per blockIdx.z (batched detection)
    cov += (size_t)blockIdx.z * 3 * w * h;
    const uint8_t* r0 = img + (long long)(y - 1) * pitch + x;
    const uint8_t* r1 = r0 + pitch;
    const uint8_t* r2 = r1 + pitch;
    const int a0 = r0[-1], a1 = r0[0], a2 = r0[1];
    const int b0 = r1[-1], b2 = r1[1];
    const int c0 = r2[-1], c1 = r2[0], c2 = r2[1];
    // Dx: symmetric column filter over exact row differences, fused as cv2's AVX2 path
    const int s0 = a2 - a0, s1 = b2 - b0, s2 = c2 - c0;
    const float dx = __fmaf_rn((float)(s0 + s2), k0, __fmul_rn((float)s1, k1));
    // Dy: smoothed rows (fused in the vectorised body, unfused in the scalar tail), then r[y+1]-r[y-1]
    float rt, rb;
    if (x < (w & ~31)) {
        rt = __fmaf_rn(k0, (float)a2, __fmaf_rn(k1, (float)a1, __fmul_rn(k0, (float)a0)));
        rb = __fmaf_rn(k0, (float)c2, __fmaf_rn(k1, (float)c1, __fmul_rn(k0, (float)c0)));
    } else {
        rt = __fadd_rn(__fadd_rn(__fmul_rn(k0, (float)a0), __fmul_rn(k1, (float)a1)), __fmul_rn(k0, (float)a2));
        rb = __fadd_rn(__fadd_rn(__fmul_rn(k0, (float)c0), __fmul_rn(k1, (float)c1)), __fmul_rn(k0, (float)c2));
    }
    const float dy = __fsub_rn(rb, rt);
    float* c = cov + 3 * ((size_t)y * w + x);
    c[0] = __fmul_rn(dx, dx); c[1] = __fmul_rn(dx, dy); c[2] = __fmul_rn(dy, dy);
}

// 3x3 box filter of the three covariance planes exactly as cv2's boxFilter<float -> double -> float>
// runs it: row sums in double, then a RUNNING column sum in double (SUM += entering row, emit,
// SUM -= leaving row) whose rounding history is part of the result -- so the sum down a column is a
// serial chain.  Split so that only the chain itself is serial:
//   gftt_colsum_kernel   one thread per (column, plane): double row sums formed on the fly + the chain, prefetching 8 rows ahead
//   gftt_eig_kernel      a + c - sqrt((a - c)^2 + b^2) and the global maximum                   (parallel)
// single-image path: parallel double row sums, then the chain with one coalesced load per step
__global__ void __launch_bounds__(256)
gftt_rowsum_kernel(const float* __restrict__ cov, int w, int h, double* __restrict__ rs)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int yy = (int)blockIdx.y - 1;
    if (x >= w) return;
    const int xm = refl101(x - 1, w), xp = refl101(x + 1, w);
    const float* r = cov + 3 * (size_t)refl101(yy, h) * w;
#pragma unroll
    for (int ch = 0; ch < 3; ++ch)
        rs[((size_t)(yy + 1) * 3 + ch) * w + x] = __dadd_rn(__dadd_rn((double)r[3 * xm + ch], (double)r[3 * x + ch]), (double)r[3 * xp + ch]);
}

__global__ void __launch_bounds__(32)
gftt_colsum_rs_kernel(const double* __restrict__ rs, int w, int h, float* __restrict__ box /* [3][h][w] */)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 3 * w) return;
    const int ch = t / w, x = t - ch * w;
    const double* col = rs + (size_t)ch * w + x;           // row yy at col[(yy + 1) * 3 * w]
    const size_t rstep = (size_t)3 * w;
    float* out = box + (size_t)ch * w * h + x;
    double prev1 = col[0], prev0 = col[rstep];
    double SUM = __dadd_rn(__dadd_rn(0., prev1), prev0);
    constexpr int RB = 8;
    double nxt[RB];
#pragma unroll
    for (int k = 0; k < RB; ++k) nxt[k] = (k + 1 <= h) ? col[(size_t)(k + 2) * rstep] : 0.;
    for (int y0 = 0; y0 < h; y0 += RB) {
        double blk[RB];
#pragma unroll
        for (int k = 0; k < RB; ++k) blk[k] = nxt[k];
#pragma unroll
        for (int k = 0; k < RB; ++k) nxt[k] = (y0 + RB + k + 1 <= h) ? col[(size_t)(y0 + RB + k + 2) * rstep] : 0.;
#pragma unroll
        for (int k = 0; k < RB; ++k) {
            const int y = y0 + k;
            if (y < h) {
                const double s0 = __dadd_rn(SUM, blk[k]);
                out[(size_t)y * w] = (float)s0;
                SUM = __dsub_rn(s0, prev1);
                prev1 = prev0; prev0 = blk[k];
            }
        }
    }
}

// one thread per (column, plane): the double row sum of each entering row is formed on the fly from the three
// neighbouring covariance values (cached: the three planes of a pixel share a line), then joins the chain
__global__ void __launch_bounds__(32)
gftt_colsum_kernel(const float* __restrict__ cov, int w, int h, float* __restrict__ box /* [3][h][w] */)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 3 * w) return;
    cov += (size_t)blockIdx.y * 3 * w * h;
    box += (size_t)blockIdx.y * 3 * w * h;
    const int x = t / 3, ch = t - x * 3;                   // the three planes of a column sit in adjacent lanes
    const int xm = refl101(x - 1, w), xp = refl101(x + 1, w);
    auto rowsum = [&](int yy) {
        const float* r = cov + 3 * (size_t)refl101(yy, h) * w + ch;
        return __dadd_rn(__dadd_rn((double)r[3 * xm], (double)r[3 * x]), (double)r[3 * xp]);
    };
    float* out = box + (size_t)ch * w * h + x;
    double prev1 = rowsum(-1), prev0 = rowsum(0);
    double SUM = __dadd_rn(__dadd_rn(0., prev1), prev0);
    constexpr int RB = 8;
    double nxt[RB];
#pragma unroll
    for (int k = 0; k < RB; ++k) nxt[k] = rowsum(k + 1);
    for (int y0 = 0; y0 < h; y0 += RB) {
        double blk[RB];
#pragma unroll
        for (int k = 0; k < RB; ++k) blk[k] = nxt[k];
        if (y0 + RB < h) {
#pragma unroll
            for (int k = 0; k < RB; ++k) nxt[k] = rowsum(y0 + RB + k + 1);
        }
#pragma unroll
        for (int k = 0; k < RB; ++k) {
            const int y = y0 + k;
            if (y < h) {
                const double s0 = __dadd_rn(SUM, blk[k]);
                out[(size_t)y * w] = (float)s0;
                SUM = __dsub_rn(s0, prev1);
                prev1 = prev0; prev0 = blk[k];
            }
        }
    }
}

// Batched path: covariance, box filter and eigenvalue in ONE pass down the columns.  A warp owns 30 adjacent
// columns (lanes 1..30; lanes 0 and 31 carry the REFLECT_101 neighbours x0-1 and x0+30).  Per image row every lane
// forms the three covariance products of its column exactly as gftt_cov_kernel does, the double row sums come from
// the neighbouring lanes by shuffle, and the three running column sums, the eigenvalue and the per-image maximum
// follow -- the covariance and box planes (24 B per pixel) never exist in memory.
#define GF_COLS 30
__global__ void __launch_bounds__(32)
gftt_fused_eig_kernel(const uint8_t* __restrict__ img, size_t img_stride, int pitch, int w, int h, float k0, float k1,
                      float* __restrict__ eig, int* __restrict__ max_bits, int small_stride, const VoSeqExt* __restrict__ ext,
                      const int* __restrict__ list)
{
    const int lane = threadIdx.x;
    const int im = list ? list[blockIdx.y] : blockIdx.y;
    img += im * img_stride;
    eig += (size_t)im * w * h;                  // planes of the slot size; a sequence's own plane has rows of its own width
    max_bits += im * small_stride;
    if (ext) {
        w = ext[im].w[0]; h = ext[im].h[0];
        if ((int)blockIdx.x * GF_COLS >= w) return;
    }
    const int xv = blockIdx.x * GF_COLS + lane - 1;            // virtual column (may be -1 or >= w)
    const int x = refl101(xv < w + 1 ? xv : w, w);              // column whose covariance this lane forms
    const bool owner = lane >= 1 && lane <= GF_COLS && xv < w;
    const bool fused_cols = x < (w & ~31);
    auto cov_row = [&](int yy, float* c) {                      // covariance products of pixel (x, refl(yy))
        const int y = refl101(yy, h);
        const uint8_t* r0 = img + (long long)(y - 1) * pitch + x;
        const uint8_t* r1 = r0 + pitch;
        const uint8_t* r2 = r1 + pitch;
        const int a0 = r0[-1], a1 = r0[0], a2 = r0[1];
        const int b0 = r1[-1], b2 = r1[1];
        const int c0 = r2[-1], c1 = r2[0], c2 = r2[1];
        const int s0 = a2 - a0, s1 = b2 - b0, s2 = c2 - c0;
        const float dx = __fmaf_rn((float)(s0 + s2), k0, __fmul_rn((float)s1, k1));
        float rt, rb;
        if (fused_cols) {
            rt = __fmaf_rn(k0, (float)a2, __fmaf_rn(k1, (float)a1, __fmul_rn(k0, (float)a0)));
            rb = __fmaf_rn(k0, (float)c2, __fmaf_rn(k1, (float)c1, __fmul_rn(k0, (float)c0)));
        } else {
            rt = __fadd_rn(__fadd_rn(__fmul_rn(k0, (float)a0), __fmul_rn(k1, (float)a1)), __fmul_rn(k0, (float)a2));
            rb = __fadd_rn(__fadd_rn(__fmul_rn(k0, (float)c0), __fmul_rn(k1, (float)c1)), __fmul_rn(k0, (float)c2));
        }
        const float dy = __fsub_rn(rb, rt);
        c[0] = __fmul_rn(dx, dx); c[1] = __fmul_rn(dx, dy); c[2] = __fmul_rn(dy, dy);
    };
    auto row_sums = [&](const float* c, double* rs) {           // double sum of the left, own and right column
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {                        // one conversion per value, the doubles travel
            const double m = (double)c[ch];
            const double l = __shfl_up_sync(0xffffffffu, m, 1), r = __shfl_down_sync(0xffffffffu, m, 1);
            rs[ch] = __dadd_rn(__dadd_rn(l, m), r);
        }
    };
    // covariance products from a 3 x 3 pixel window held in registers (a*: row above, b*: own row, c*: row below)
    auto cov_win = [&](int a0, int a1, int a2, int b0, int b2, int c0, int c1, int c2, float* c) {
        const int s0 = a2 - a0, s1 = b2 - b0, s2 = c2 - c0;
        const float dx = __fmaf_rn((float)(s0 + s2), k0, __fmul_rn((float)s1, k1));
        float rt, rb;
        if (fused_cols) {
            rt = __fmaf_rn(k0, (float)a2, __fmaf_rn(k1, (float)a1, __fmul_rn(k0, (float)a0)));
            rb = __fmaf_rn(k0, (float)c2, __fmaf_rn(k1, (float)c1, __fmul_rn(k0, (float)c0)));
        } else {
            rt = __fadd_rn(__fadd_rn(__fmul_rn(k0, (float)a0), __fmul_rn(k1, (float)a1)), __fmul_rn(k0, (float)a2));
            rb = __fadd_rn(__fadd_rn(__fmul_rn(k0, (float)c0), __fmul_rn(k1, (float)c1)), __fmul_rn(k0, (float)c2));
        }
        const float dy = __fsub_rn(rb, rt);
        c[0] = __fmul_rn(dx, dx); c[1] = __fmul_rn(dx, dy); c[2] = __fmul_rn(dy, dy);
    };
    float c[3];
    double prev1[3], prev0[3], SUM[3];
    cov_row(-1, c); row_sums(c, prev1);       // leaving row of y = 0: image row 1
    cov_row(0, c); row_sums(c, prev0);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) SUM[ch] = __dadd_rn(__dadd_rn(0., prev1[ch]), prev0[ch]);
    float vmax = 0.f;
    // Entering rows yy = 1 .. h-1 are consecutive image rows: a sliding window needs three new pixels per row.
    // The pixel triples of the next RB rows are fetched while the chain of this block runs.  The last entering
    // row (yy = h) is image row h-2 again and is formed on its own.
    const uint8_t* prow = img + x;                                   // pixel (x, 0); rows -1 .. h exist (border)
    int w0[3], w1[3], w2[3];                                         // window rows: (yy-1), yy, (yy+1) for the row being formed
    {
        const uint8_t* r = prow;                                     // row 0
        w0[0] = r[-1]; w0[1] = r[0]; w0[2] = r[1];
        r += pitch;                                                  // row 1
        w1[0] = r[-1]; w1[1] = r[0]; w1[2] = r[1];
    }
    constexpr int RB = 8;
    int nx0[RB], nx1[RB], nx2[RB];
    auto fetch = [&](int yy_first) {                                 // pixel rows yy_first+1 .. yy_first+RB (the row BELOW each entering row)
#pragma unroll
        for (int k = 0; k < RB; ++k) {
            const int pr = min(yy_first + k + 1, h);                 // row h is the materialised border row
            const uint8_t* r = prow + (long long)pr * pitch;
            nx0[k] = r[-1]; nx1[k] = r[0]; nx2[k] = r[1];
        }
    };
    fetch(1);
    auto emit = [&](int y, const float* cv) {                        // entering row formed: advance the three chains, write eig(y)
        double cur[3];
        row_sums(cv, cur);
        float bx[3];
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const double s0 = __dadd_rn(SUM[ch], cur[ch]);
            bx[ch] = (float)s0;
            SUM[ch] = __dsub_rn(s0, prev1[ch]);
            prev1[ch] = prev0[ch]; prev0[ch] = cur[ch];
        }
        const float a = __fmul_rn(bx[0], 0.5f), b = bx[1], cc = __fmul_rn(bx[2], 0.5f);
        const float t = __fsub_rn(a, cc);
        const float v = __fsub_rn(__fadd_rn(a, cc), __fsqrt_rn(__fadd_rn(__fmul_rn(t, t), __fmul_rn(b, b))));
        if (owner) { eig[(size_t)y * w + xv] = v; vmax = fmaxf(vmax, v); }
    };
    for (int yy0 = 1; yy0 <= h - 1; yy0 += RB) {                     // entering rows yy0 .. yy0+RB-1 (output rows yy-1)
        int b0[RB], b1[RB], b2[RB];
#pragma unroll
        for (int k = 0; k < RB; ++k) { b0[k] = nx0[k]; b1[k] = nx1[k]; b2[k] = nx2[k]; }
        if (yy0 + RB <= h - 1) fetch(yy0 + RB);
#pragma unroll
        for (int k = 0; k < RB; ++k) {
            const int yy = yy0 + k;
            if (yy <= h - 1) {                                       // warp-uniform
                float cv[3];
                cov_win(w0[0], w0[1], w0[2], w1[0], w1[2], b0[k], b1[k], b2[k], cv);
                emit(yy - 1, cv);
                w0[0] = w1[0]; w0[1] = w1[1]; w0[2] = w1[2];
                w1[0] = b0[k]; w1[1] = b1[k]; w1[2] = b2[k];
            }
        }
    }
    cov_row(h, c);                                                   // last entering row: image row h-2
    emit(h - 1, c);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if (lane == 0 && vmax > __int_as_float(*(volatile int*)max_bits)) atomicMax(max_bits, __float_as_int(vmax));
}

__global__ void __launch_bounds__(256)
gftt_eig_kernel(const float* __restrict__ box, int w, int h, float* __restrict__ eig, int* __restrict__ max_bits, int small_stride)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, npx = (size_t)w * h;
    box += (size_t)blockIdx.y * 3 * npx;
    eig += (size_t)blockIdx.y * npx;
    max_bits += blockIdx.y * small_stride;
    float v = 0.f;
    if (i < npx) {
        const float a = __fmul_rn(box[i], 0.5f), b = box[npx + i], c = __fmul_rn(box[2 * npx + i], 0.5f);
        const float t = __fsub_rn(a, c);
        v = __fsub_rn(__fadd_rn(a, c), __fsqrt_rn(__fadd_rn(__fmul_rn(t, t), __fmul_rn(b, b))));
        eig[i] = v;
    }
    // eig >= 0 up to rounding; negative values never win the max (cv2's max would be >= 0 too).
    // One atomic per CTA, and only when it can raise the running maximum (a batch has 64 hot addresses).
    __shared__ float s_max[8];
    float vmax = fmaxf(v, 0.f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = vmax;
    __syncthreads();
    if (threadIdx.x == 0) {
        float m = s_max[0];
#pragma unroll
        for (int k = 1; k < 8; ++k) m = fmaxf(m, s_max[k]);
        if (m > __int_as_float(*(volatile int*)max_bits)) atomicMax(max_bits, __float_as_int(m));
    }
}

__global__ void __launch_bounds__(256)
gftt_candidates_kernel(const float* __restrict__ eig, int w, int h, const int* __restrict__ max_bits, double quality,
                       unsigned long long* __restrict__ keys, int* __restrict__ n_keys, int cap, int small_stride,
                       const VoSeqExt* __restrict__ ext = nullptr, const int* __restrict__ list = nullptr)
{
    const int im = list ? list[blockIdx.z] : blockIdx.z;
    eig += (size_t)im * w * h;
    if (ext) { w = ext[im].w[0]; h = ext[im].h[0]; }   // key address y * w + x: cv2's tie order in its own image
    max_bits += im * small_stride;
    n_keys += im * small_stride;
    keys += (size_t)im * cap;
    const int x = blockIdx.x * blockDim.x + threadIdx.x + 1;
    const float thr = (float)((double)__int_as_float(*max_bits) * quality);
    const int lane = (threadIdx.y * blockDim.x + threadIdx.x) & 31;
#pragma unroll
    for (int k = 0; k < 4; ++k) {                        // a 32 x 8 block covers 32 x 32 pixels: four rows per thread
        const int y = blockIdx.y * 32 + 8 * k + threadIdx.y + 1;
        bool is_c = false;
        float v = 0.f;
        if (x < w - 1 && y < h - 1) {
            const float* p = eig + (size_t)y * w + x;
            v = p[0];
            if (v > thr)
                is_c = !(p[-w - 1] > v || p[-w] > v || p[-w + 1] > v || p[-1] > v || p[1] > v || p[w - 1] > v || p[w] > v || p[w + 1] > v);
        }
        const unsigned m = __ballot_sync(0xffffffffu, is_c);
        if (!m) continue;
        int base = 0;
        if (lane == __ffs(m) - 1) base = atomicAdd(n_keys, __popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (is_c) {
            const int pos = base + __popc(m & ((1u << lane) - 1));
            if (pos < cap) keys[pos] = ((unsigned long long)__float_as_uint(v) << 32) | (unsigned)(y * w + x);
        }
    }
}

// descending order of the 64-bit keys = (value desc, address desc); keys are unique
__global__ void __launch_bounds__(256)
gftt_rank_kernel(const unsigned long long* __restrict__ keys, const int* __restrict__ n_keys, int cap,
                 unsigned long long* __restrict__ sorted, int small_stride, const int* __restrict__ list = nullptr)
{
    __shared__ unsigned long long tile[1024];
    const int im = list ? list[blockIdx.y] : blockIdx.y;
    keys += (size_t)im * cap;
    sorted += (size_t)im * cap;
    n_keys += im * small_stride;
    const int n = min(*n_keys, cap);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x * blockDim.x >= n) return;
    const unsigned long long mine = i < n ? keys[i] : 0ull;
    int rank = 0;
    for (int t0 = 0; t0 < n; t0 += 1024) {
        __syncthreads();
        for (int k = threadIdx.x; k < 1024; k += blockDim.x) tile[k] = (t0 + k < n) ? keys[t0 + k] : 0ull;
        __syncthreads();
        const int lim = min(1024, n - t0);
#pragma unroll 8
        for (int k = 0; k < lim; ++k) rank += tile[k] > mine;
    }
    if (i < n) sorted[rank] = mine;
}

// bitonic sort (descending) in global memory for large candidate sets; n_pad = power of two
__global__ void gftt_bitonic_pad_kernel(unsigned long long* keys, const int* n_keys, int cap, int n_pad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = min(*n_keys, cap);
    if (i < n_pad && i >= n) keys[i] = 0ull;
}
__global__ void gftt_bitonic_step_kernel(unsigned long long* keys, int j, int k, int n_pad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    const int l = i ^ j;
    if (l > i) {
        const unsigned long long a = keys[i], b = keys[l];
        const bool desc = (i & k) == 0;
        if (desc ? (a < b) : (a > b)) { keys[i] = b; keys[l] = a; }
    }
}

#define GFTT_CELL_CAP 8
// single warp; grid cells hold accepted corners (x | y << 16)
__global__ void __launch_bounds__(32)
gftt_select_kernel(const unsigned long long* __restrict__ sorted, const int* __restrict__ n_keys, int cap, int w, int h,
                   int max_corners, double min_dist, int cell, int gw, int gh, int* __restrict__ cell_cnt,
                   int* __restrict__ cell_pts, float* __restrict__ corners, int* __restrict__ n_out)
{
    const int lane = threadIdx.x;
    const int n = min(*n_keys, cap);
    const double md2 = min_dist * min_dist;
    int n_acc = 0;
    const int limit = max_corners > 0 ? max_corners : 0x7fffffff;
    if (min_dist < 1) {
        const int m = min(n, limit);
        for (int i = lane; i < m; i += 32) {
            const int idx = (int)(sorted[i] & 0xffffffffu);
            corners[2 * i] = (float)(idx % w); corners[2 * i + 1] = (float)(idx / w);
        }
        if (lane == 0) *n_out = m;
        return;
    }
    for (int i0 = 0; i0 < n && n_acc < limit; i0 += 32) {
        const int i = i0 + lane;
        int x = 0, y = 0;
        bool alive = i < n;
        if (alive) {
            const int idx = (int)(sorted[i] & 0xffffffffu);
            y = idx / w; x = idx - y * w;
            const int xc = x / cell, yc = y / cell;
            const int x1 = max(0, xc - 1), y1 = max(0, yc - 1), x2 = min(gw - 1, xc + 1), y2 = min(gh - 1, yc + 1);
            for (int yy = y1; yy <= y2 && alive; ++yy)
                for (int xx = x1; xx <= x2 && alive; ++xx) {
                    const int c = yy * gw + xx;
                    const int cnt = __ldcg(cell_cnt + c);
                    for (int j = 0; j < cnt; ++j) {
                        const int p = __ldcg(cell_pts + c * GFTT_CELL_CAP + j);
                        const float dx = (float)(x - (p & 0xffff)), dy = (float)(y - (p >> 16));
                        if ((double)(dx * dx + dy * dy) < md2) { alive = false; break; }
                    }
                }
        }
        // survivors of this chunk: accept in order, each acceptance kills later survivors within min_dist
        unsigned surv = __ballot_sync(0xffffffffu, alive);
        while (surv && n_acc < limit) {
            const int f = __ffs(surv) - 1;
            const int fx = __shfl_sync(0xffffffffu, x, f), fy = __shfl_sync(0xffffffffu, y, f);
            if (lane == f) {
                const int c = (y / cell) * gw + (x / cell);
                const int cnt = cell_cnt[c];
                if (cnt < GFTT_CELL_CAP) { cell_pts[c * GFTT_CELL_CAP + cnt] = x | (y << 16); cell_cnt[c] = cnt + 1; }
                corners[2 * n_acc] = (float)x; corners[2 * n_acc + 1] = (float)y;
                alive = false;
            }
            ++n_acc;
            if (alive) {
                const float dx = (float)(x - fx), dy = (float)(y - fy);
                if ((double)(dx * dx + dy * dy) < md2) alive = false;
            }
            surv = __ballot_sync(0xffffffffu, alive);
        }
        __threadfence_block();
        __syncwarp();
    }
    if (lane == 0) *n_out = n_acc;
}

// Same greedy selection with the cell grid in shared memory (16 B per cell: up to four accepted
// corners as x | y << 16, ~0 = empty -- corners of one cell are pairwise >= min_dist apart, a
// cell is round(min_dist) wide, so at most two or three ever share one).  256 threads clear the
// grid, one warp runs the selection; every neighbourhood test is nine independent LDS.128.
#define GFTT_SCELL_CAP 4
__global__ void __launch_bounds__(256)
gftt_select_smem_kernel(const unsigned long long* __restrict__ sorted, const int* __restrict__ n_keys, int cap, int w, int h,
                        int max_corners, double min_dist, int cell, int gw, int gh, float* __restrict__ corners,
                        int* __restrict__ n_out, int small_stride, size_t out_stride, const VoSeqExt* __restrict__ ext = nullptr,
                        const int* __restrict__ list = nullptr)
{
    extern __shared__ uint4 s_cells[];
    const int im = list ? list[blockIdx.x] : blockIdx.x;   // one CTA per image
    if (ext) {   // the image's own cell grid (the shared memory is sized for the slot's)
        w = ext[im].w[0]; h = ext[im].h[0];
        gw = (w + cell - 1) / cell; gh = (h + cell - 1) / cell;
    }
    sorted += (size_t)im * cap;
    n_keys += im * small_stride;
    n_out += im * small_stride;
    corners += im * out_stride;
    for (int i = threadIdx.x; i < gw * gh; i += blockDim.x) s_cells[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
    __syncthreads();
    if (threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    const int n = min(*n_keys, cap);
    const double md2 = min_dist * min_dist;
    int n_acc = 0;
    const int limit = max_corners > 0 ? max_corners : 0x7fffffff;
    unsigned long long key_next = lane < n ? sorted[lane] : 0ull;
    for (int i0 = 0; i0 < n && n_acc < limit; i0 += 32) {
        const int i = i0 + lane;
        int x = 0, y = 0;
        bool alive = i < n;
        const unsigned long long key = key_next;
        if (i + 32 < n) key_next = sorted[i + 32];      // the next chunk's keys travel while this chunk is resolved
        if (alive) {
            const int idx = (int)(key & 0xffffffffu);
            y = idx / w; x = idx - y * w;
            const int xc = x / cell, yc = y / cell;
#pragma unroll
            for (int dyc = -1; dyc <= 1; ++dyc)
#pragma unroll
                for (int dxc = -1; dxc <= 1; ++dxc) {
                    const int xx = xc + dxc, yy = yc + dyc;
                    if (xx < 0 || yy < 0 || xx >= gw || yy >= gh) continue;
                    const uint4 c = s_cells[yy * gw + xx];
                    const unsigned pv[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
                    for (int j = 0; j < GFTT_SCELL_CAP; ++j) {
                        if (pv[j] == ~0u) continue;
                        const float dx = (float)(x - (int)(pv[j] & 0xffff)), dy = (float)(y - (int)(pv[j] >> 16));
                        if ((double)(dx * dx + dy * dy) < md2) alive = false;
                    }
                }
        }
        // survivors of this chunk, in priority order: a survivor is accepted iff no ACCEPTED earlier
        // survivor of the chunk lies within min_dist.  Every lane first collects the bit mask of earlier
        // survivors in conflict with it (32 independent shuffles), then the acceptance recurrence runs
        // on bit masks, identically in every lane (one shuffle per survivor instead of a ballot loop).
        const unsigned surv = __ballot_sync(0xffffffffu, alive);
        unsigned accepted = 0;
        if (surv) {
            unsigned conf = 0;
#pragma unroll
            for (int f = 0; f < 32; ++f) {          // 64 independent shuffles, fully pipelined
                const int fx = __shfl_sync(0xffffffffu, x, f), fy = __shfl_sync(0xffffffffu, y, f);
                const float dx = (float)(x - fx), dy = (float)(y - fy);
                if (f < lane && ((surv >> f) & 1u) && (double)(dx * dx + dy * dy) < md2) conf |= 1u << f;
            }
            unsigned cf[32];
#pragma unroll
            for (int f = 0; f < 32; ++f) cf[f] = __shfl_sync(0xffffffffu, conf, f);
            int room = limit - n_acc;
#pragma unroll
            for (int f = 0; f < 32; ++f)
                if (((surv >> f) & 1u) && !(cf[f] & accepted) && room > 0) { accepted |= 1u << f; --room; }
        }
        if ((accepted >> lane) & 1u) {
            const int o = n_acc + __popc(accepted & ((1u << lane) - 1));
            corners[2 * o] = (float)x; corners[2 * o + 1] = (float)y;
            unsigned* cp = reinterpret_cast<unsigned*>(&s_cells[(y / cell) * gw + (x / cell)]);
            const unsigned val = (unsigned)x | ((unsigned)y << 16);
#pragma unroll
            for (int j = 0; j < GFTT_SCELL_CAP; ++j)
                if (atomicCAS(cp + j, ~0u, val) == ~0u) break;
        }
        n_acc += __popc(accepted);
        __syncwarp();
    }
    if (lane == 0) *n_out = n_acc;
}

extern "C" int b200vo_good_features_to_track(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols, size_t step,
                                             int max_corners, double quality, double min_dist, int block_size,
                                             float* corners_xy, int* n_out)
{
    if (!ctx || !img || !corners_xy || !n_out) return B200VO_E_BADARG;
    *n_out = 0;
    if (!(quality > 0) || min_dist < 0 || max_corners < 0)   // cv2: featureselect.cpp CV_Assert
        return vo_set_err(ctx, B200VO_E_BADARG, "qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0");
    if (block_size != 3) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "blockSize != 3 not implemented (the reference uses 3)");
    if (rows < 3 || cols < 3 || cols >= 65536 || rows >= 32768) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "image size");
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const int w = cols, h = rows;
    const size_t npx = (size_t)w * h;
    // bordered level 0 in the internal slot
    FrameSlot& fs = ctx->slots[B200VO_MAX_SLOTS + 1];
    PyrGeom g;
    vo_pyr_geom(rows, cols, 1, &g);
    VO_TRY(vo_reserve(ctx, fs.slab, g.slab_bytes));
    fs.valid = false;
    VO_TRY(vo_reserve(ctx, ctx->d_stage_img[1], npx));
    VO_TRY(vo_reserve_pinned(ctx, vo_align(npx, 256) + 4096));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    if (step == (size_t)cols) memcpy(hp, img, npx);
    else for (int y = 0; y < rows; ++y) memcpy(hp + (size_t)y * cols, img + (size_t)y * step, (size_t)cols);
    VO_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage_img[1].p, hp, npx, cudaMemcpyHostToDevice, ctx->stream));
    VO_TRY(vo_build_pyramids(ctx, (const uint8_t*)ctx->d_stage_img[1].p, npx, rows, cols, g, (uint8_t*)fs.slab.p, g.slab_bytes, 1, ctx->stream));
    const uint8_t* d_img = (const uint8_t*)fs.slab.p + g.off[0];
    // scratch: cov | eig | keys | sorted | cells | small
    const int cell = min_dist >= 1 ? (int)llrint(min_dist) : 1;
    const int gw = (w + cell - 1) / cell, gh = (h + cell - 1) / cell;
    const int cap = (int)npx;
    int n_pad = 1;
    while (n_pad < cap) n_pad <<= 1;
    const size_t b_cov = vo_align(npx * 12, 256), b_eig = vo_align(npx * 4, 256), b_keys = vo_align((size_t)n_pad * 8, 256);
    const size_t b_cnt = vo_align((size_t)gw * gh * 4, 256), b_pts = vo_align((size_t)gw * gh * GFTT_CELL_CAP * 4, 256);
    const size_t out_cap = max_corners > 0 ? (size_t)max_corners : npx;
    const size_t b_out = vo_align(out_cap * 8, 256), b_small = 256;
    const size_t b_rs = vo_align((size_t)(h + 2) * 3 * w * 8, 256), b_box = vo_align(npx * 12, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[2], b_cov + b_eig + 2 * b_keys + b_cnt + b_pts + b_out + b_small + b_rs + b_box));
    uint8_t* d = (uint8_t*)ctx->d_scratch[2].p;
    double* d_rs = (double*)(d + b_cov + b_eig + 2 * b_keys + b_cnt + b_pts + b_out + b_small);
    float* d_box = (float*)((uint8_t*)d_rs + b_rs);
    float* d_cov = (float*)d; d += b_cov;
    float* d_eig = (float*)d; d += b_eig;
    unsigned long long* d_keys = (unsigned long long*)d; d += b_keys;
    unsigned long long* d_sorted = (unsigned long long*)d; d += b_keys;
    int* d_cnt = (int*)d; d += b_cnt;
    int* d_pts = (int*)d; d += b_pts;
    float* d_out = (float*)d; d += b_out;
    int* d_small = (int*)d;   // [0] max bits, [1] n_keys, [2] n_out
    VO_CUDA(ctx, cudaMemsetAsync(d_small, 0, b_small, ctx->stream));
    VO_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, b_cnt, ctx->stream));
    const double scale = 1.0 / (4.0 * block_size * 255.0);
    {
        dim3 blk(32, 8), grd((w + 31) / 32, (h + 7) / 8);
        gftt_cov_kernel<<<grd, blk, 0, ctx->stream>>>(d_img, 0, g.pitch[0], w, h, (float)scale, (float)(2.0 * scale), d_cov);
        gftt_rowsum_kernel<<<dim3((w + 255) / 256, h + 2), 256, 0, ctx->stream>>>(d_cov, w, h, d_rs);
        gftt_colsum_rs_kernel<<<(3 * w + 31) / 32, 32, 0, ctx->stream>>>(d_rs, w, h, d_box);
        gftt_eig_kernel<<<(int)((npx + 255) / 256), 256, 0, ctx->stream>>>(d_box, w, h, d_eig, d_small, 0);
        ctx->launches += 2;
        dim3 grd2((w - 2 + 31) / 32, (h - 2 + 31) / 32);
        gftt_candidates_kernel<<<grd2, blk, 0, ctx->stream>>>(d_eig, w, h, d_small, quality, d_keys, d_small + 1, cap, 0);
        ctx->launches += 3;
    }
    // the candidate count decides the sort; reading it back costs one small sync (the call is synchronous anyway)
    int* h_small = (int*)(hp + vo_align(npx, 256));
    VO_CUDA(ctx, cudaMemcpyAsync(h_small, d_small, 16, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int n_keys = h_small[1] < cap ? h_small[1] : cap;
    if (n_keys == 0) { *n_out = 0; return 0; }
    const unsigned long long* d_order = d_sorted;
    if (n_keys <= 32768) {
        gftt_rank_kernel<<<(n_keys + 255) / 256, 256, 0, ctx->stream>>>(d_keys, d_small + 1, cap, d_sorted, 0);
        ctx->launches++;
    } else {
        int np = 1;
        while (np < n_keys) np <<= 1;
        gftt_bitonic_pad_kernel<<<(np + 255) / 256, 256, 0, ctx->stream>>>(d_keys, d_small + 1, cap, np);
        for (int k = 2; k <= np; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                gftt_bitonic_step_kernel<<<(np + 255) / 256, 256, 0, ctx->stream>>>(d_keys, j, k, np);
                ctx->launches++;
            }
        d_order = d_keys;
    }
    const size_t cell_smem = (size_t)gw * gh * sizeof(uint4);
    if (min_dist >= 1 && cell_smem <= 200 * 1024) {
        if (cell_smem > 48 * 1024)
            VO_CUDA(ctx, cudaFuncSetAttribute(gftt_select_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cell_smem));
        gftt_select_smem_kernel<<<1, 256, cell_smem, ctx->stream>>>(d_order, d_small + 1, cap, w, h, max_corners, min_dist, cell, gw,
                                                                    gh, d_out, d_small + 2, 0, 0);
    } else {
        gftt_select_kernel<<<1, 32, 0, ctx->stream>>>(d_order, d_small + 1, cap, w, h, max_corners, min_dist, cell, gw, gh, d_cnt,
                                                      d_pts, d_out, d_small + 2);
    }
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    VO_CUDA(ctx, cudaMemcpyAsync(h_small, d_small, 16, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const int n = h_small[2];
    if (n > 0) {
        VO_TRY(vo_reserve_pinned(ctx, (size_t)n * 8 + 4096));
        VO_CUDA(ctx, cudaMemcpyAsync(ctx->h_pin, d_out, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
        memcpy(corners_xy, ctx->h_pin, (size_t)n * 8);
    }
    *n_out = n;
    return 0;
}

// Batched detection on device-resident bordered level-0 images (one per sequence, `img_stride` bytes apart):
// every kernel above with the image index in the grid, one selection CTA per image, no intermediate host
// synchronisation (at most GFTT_BATCH_CAP candidates per image, ranked by counting).
#define GFTT_BATCH_CAP VO_GFTT_BATCH_CAP
#define GFTT_SMALL VO_GFTT_SMALL

size_t vo_gftt_batch_workspace(int rows, int cols, int batch, int max_corners)
{
    const size_t npx = (size_t)rows * cols;
    return vo_align(npx * 4 * batch, 256) +
           (size_t)batch * (2 * vo_align((size_t)GFTT_BATCH_CAP * 8, 256) + vo_align((size_t)max_corners * 8, 256)) +
           vo_align((size_t)batch * GFTT_SMALL * sizeof(int), 256);
}

int vo_gftt_batch_launch(b200vo_ctx* ctx, const uint8_t* d_img0, size_t img_stride, int pitch, int rows, int cols, int batch,
                         int max_corners, double quality, double min_dist, void* ws, float** d_corners_out, int** d_small_out,
                         const VoSeqExt* d_ext, const int* d_list, int n_img)
{
    const int w = cols, h = rows;
    if (!d_list) n_img = batch;
    const size_t npx = (size_t)w * h;
    if (!(quality > 0) || min_dist < 0 || max_corners < 0)
        return vo_set_err(ctx, B200VO_E_BADARG, "qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0");
    const int cell = (int)llrint(min_dist);
    const int gw = cell > 0 ? (w + cell - 1) / cell : 0, gh = cell > 0 ? (h + cell - 1) / cell : 0;
    const size_t cell_smem = (size_t)gw * gh * sizeof(uint4);
    if (min_dist < 1 || max_corners <= 0 || cell_smem > 200 * 1024 || rows < 3 || cols < 3 || cols >= 65536 || rows >= 32768)
        return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "batched detection needs minDistance >= 1, maxCorners > 0 and a cell grid that fits shared memory");
    // per-image planes are tightly packed (the kernels derive the image offsets from w, h)
    const size_t b_keys = vo_align((size_t)GFTT_BATCH_CAP * 8, 256), b_out = vo_align((size_t)max_corners * 8, 256);
    uint8_t* d = (uint8_t*)ws;
    float* d_eig = (float*)d; d += vo_align(npx * 4 * batch, 256);
    unsigned long long* d_keys = (unsigned long long*)d; d += b_keys * batch;
    unsigned long long* d_sorted = (unsigned long long*)d; d += b_keys * batch;
    float* d_out = (float*)d; d += b_out * batch;
    int* d_small = (int*)d;
    VO_CUDA(ctx, cudaMemsetAsync(d_small, 0, (size_t)batch * GFTT_SMALL * sizeof(int), ctx->stream));
    const double scale = 1.0 / (4.0 * 3 * 255.0);
    dim3 blk(32, 8);
    gftt_fused_eig_kernel<<<dim3((w + GF_COLS - 1) / GF_COLS, n_img), 32, 0, ctx->stream>>>(d_img0, img_stride, pitch, w, h, (float)scale,
                                                                                            (float)(2.0 * scale), d_eig, d_small, GFTT_SMALL, d_ext,
                                                                                            d_list);
    gftt_candidates_kernel<<<dim3((w - 2 + 31) / 32, (h - 2 + 31) / 32, n_img), blk, 0, ctx->stream>>>(d_eig, w, h, d_small, quality, d_keys,
                                                                                                    d_small + 1, GFTT_BATCH_CAP, GFTT_SMALL, d_ext,
                                                                                                    d_list);
    gftt_rank_kernel<<<dim3(GFTT_BATCH_CAP / 256, n_img), 256, 0, ctx->stream>>>(d_keys, d_small + 1, GFTT_BATCH_CAP, d_sorted, GFTT_SMALL,
                                                                                 d_list);
    if (cell_smem > 48 * 1024)
        VO_CUDA(ctx, cudaFuncSetAttribute(gftt_select_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cell_smem));
    gftt_select_smem_kernel<<<n_img, 256, cell_smem, ctx->stream>>>(d_sorted, d_small + 1, GFTT_BATCH_CAP, w, h, max_corners, min_dist, cell,
                                                                    gw, gh, d_out, d_small + 2, GFTT_SMALL, b_out / 4, d_ext, d_list);
    ctx->launches += 4;
    VO_CUDA(ctx, cudaGetLastError());
    *d_corners_out = d_out;
    *d_small_out = d_small;
    return 0;
}

// Device-pointer form of b200vo_good_features_to_track (SURVEY 8b `_dev`): the image is already in device memory, the
// corner list stays there.  Runs the batched pipeline for one image (no intermediate host synchronisation):
// needs minDistance >= 1, maxCorners > 0 and at most VO_GFTT_BATCH_CAP candidates above the quality threshold.
// corners_dev float32 (max_corners, 2); n_out_dev int32[1] = corners found, or -1 when the candidate limit was exceeded.
__global__ void gftt_export_kernel(const float* __restrict__ src, const int* __restrict__ small, int max_corners,
                                   float* __restrict__ dst, int* __restrict__ n_out)
{
    const bool over = small[1] > GFTT_BATCH_CAP;
    const int n = over ? 0 : small[2];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 2 * max_corners; i += gridDim.x * blockDim.x) dst[i] = i < 2 * n ? src[i] : 0.f;
    if (blockIdx.x == 0 && threadIdx.x == 0) *n_out = over ? -1 : n;
}

extern "C" int b200vo_good_features_to_track_dev(b200vo_ctx* ctx, const uint8_t* img_dev, int rows, int cols, size_t step,
                                                 int max_corners, double quality, double min_dist, int block_size,
                                                 float* corners_dev, int32_t* n_out_dev)
{
    if (!ctx || !img_dev || !corners_dev || !n_out_dev) return B200VO_E_BADARG;
    if (!(quality > 0) || min_dist < 0 || max_corners < 0)   // cv2: featureselect.cpp CV_Assert
        return vo_set_err(ctx, B200VO_E_BADARG, "qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0");
    if (block_size != 3) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "blockSize != 3 not implemented (the reference uses 3)");
    if (step < (size_t)cols) return vo_set_err(ctx, B200VO_E_BADARG, "step < cols");
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    FrameSlot& fs = ctx->slots[B200VO_MAX_SLOTS + 1];
    PyrGeom g;
    vo_pyr_geom(rows, cols, 1, &g);
    VO_TRY(vo_reserve(ctx, fs.slab, g.slab_bytes));
    fs.valid = false;
    const size_t npx = (size_t)rows * cols;
    const uint8_t* raw = img_dev;
    if (step != (size_t)cols) {
        VO_TRY(vo_reserve(ctx, ctx->d_stage_img[1], npx));
        VO_CUDA(ctx, cudaMemcpy2DAsync(ctx->d_stage_img[1].p, (size_t)cols, img_dev, step, (size_t)cols, (size_t)rows,
                                       cudaMemcpyDeviceToDevice, ctx->stream));
        raw = (const uint8_t*)ctx->d_stage_img[1].p;
    }
    VO_TRY(vo_build_pyramids(ctx, raw, npx, rows, cols, g, (uint8_t*)fs.slab.p, g.slab_bytes, 1, ctx->stream));
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[2], vo_gftt_batch_workspace(rows, cols, 1, max_corners > 0 ? max_corners : 1)));
    float* d_out = nullptr;
    int* d_small = nullptr;
    VO_TRY(vo_gftt_batch_launch(ctx, (const uint8_t*)fs.slab.p + g.off[0], g.slab_bytes, g.pitch[0], rows, cols, 1, max_corners, quality,
                                min_dist, ctx->d_scratch[2].p, &d_out, &d_small));
    gftt_export_kernel<<<(2 * max_corners + 255) / 256, 256, 0, ctx->stream>>>(d_out, d_small, max_corners, corners_dev, n_out_dev);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}
