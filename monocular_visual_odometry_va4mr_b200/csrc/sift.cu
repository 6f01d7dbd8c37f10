// SIFT detect + describe (SURVEY 8f row f4; replaces cv2.SIFT_create().detectAndCompute(img, None) at reference
// VisualOdometryPipeLine.py:35, :226-227 -- default parameters: nOctaveLayers 3, contrastThreshold 0.04, edgeThreshold 10,
// sigma 1.6, image doubled first, float32 descriptors).
//
// Parity design: OpenCV's sub-pixel refinement differentiates the DoG images twice, so one ulp of a Gaussian image moves
// a keypoint by ~1e-5 px -- the pyramid has to be bit-equal, not close.  The blur kernels therefore apply the taps in
// the order and with the FMA pattern of OpenCV's float32 row / column filters (row: ascending taps, fused for
// x < (cols & ~3); column: centre first, then symmetric pairs, fused for x < (cols & ~7)), the 3x3 solve uses the
// contraction GCC applies to sift.simd.hpp, and the orientation / descriptor histograms are accumulated in raster order
// (samples are evaluated in parallel, each histogram bin is summed by the one thread that owns it, in sample order).
// exp / cos / sin / 2^x are the double-precision routines rounded to float (OpenCV: IPP / libm float routines, correctly
// rounded in all but a few cases).  Everything is compiled with --fmad=false; FMAs are explicit.
//
// Stages: doubled image -> base blur -> per octave: 5 blurs (row pass, column pass writing the Gaussian image and the DoG
// image), nearest-neighbour halving -> extrema + refinement (one thread per DoG pixel) -> orientation histograms (one
// CTA per extremum) -> device merge sort in cv2's KeyPointsFilter::removeDuplicatedSorted order and duplicate removal
// (one CTA per frame) -> descriptors of the ordered list (one CTA per keypoint).
// Every stage runs for a chunk of same-sized frames at once: the frame index is part of the grid, each frame owns one
// block of the workspace, extrema and keypoints carry their frame.  One frame is the chunk of one.
#include "internal.cuh"
#include "sift.cuh"
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>
#include <cub/device/device_merge_sort.cuh>

#define SIFT_LAYERS 3
#define SIFT_IMG_BORDER 5
#define SIFT_MAX_INTERP_STEPS 5
#define SIFT_ORI_BINS 36
#define SIFT_MAX_TAPS 32
#define SIFT_MAX_OCTAVES 16

struct SiftTaps { float k[SIFT_MAX_TAPS]; int n; };

struct SiftCand {        // an extremum that survived the refinement
    float x, y, size, response;
    int octave_code;     // cv2's packed octave field, before the firstOctave shift
    int o, layer, r, c;  // pyramid octave index, refined layer, refined integer position
    int f;               // frame of the chunk
};

struct SiftKp {          // a keypoint (extremum + one orientation)
    float x, y, size, angle, response;
    int octave_code;
    int o, layer;
    int f;               // frame of the chunk; -1: a slot freed by the duplicate removal
};

__device__ __forceinline__ int sift_reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}
__device__ __forceinline__ int sift_floor(float v) { const int i = (int)v; return i - (i > v); }
__device__ __forceinline__ float sift_exp(float x) { return (float)exp((double)x); }

// ---------------------------------------------------------------- image doubling (resize INTER_LINEAR, weights 0.25 / 0.75)
__global__ void __launch_bounds__(256)
sift_upscale_kernel(const uint8_t* __restrict__ img, int rows, int cols, size_t step, size_t img_stride, float* __restrict__ out,
                    size_t fstride)
{
    const int dx = blockIdx.x * blockDim.x + threadIdx.x, dy = blockIdx.y;
    img += blockIdx.z * img_stride;
    out += blockIdx.z * fstride;
    if (dx >= 2 * cols) return;
    float fx = (float)((dx + 0.5) * 0.5 - 0.5);
    int sx = sift_floor(fx);
    fx -= sx;
    if (sx < 0) { fx = 0; sx = 0; }
    if (sx >= cols - 1) { fx = 0; sx = cols - 1; }
    float fy = (float)((dy + 0.5) * 0.5 - 0.5);
    int sy = sift_floor(fy);
    fy -= sy;
    if (sy < 0) { fy = 0; sy = 0; }
    if (sy >= rows - 1) { fy = 0; sy = rows - 1; }
    const uint8_t* r0 = img + (size_t)sy * step;
    const uint8_t* r1 = img + (size_t)(sy + 1 < rows ? sy + 1 : sy) * step;
    const int x1 = sx + 1 < cols ? sx + 1 : sx;
    const float h0 = (float)r0[sx] * (1.f - fx) + (float)r0[x1] * fx;
    const float h1 = (float)r1[sx] * (1.f - fx) + (float)r1[x1] * fx;
    out[(size_t)dy * (2 * cols) + dx] = h0 * (1.f - fy) + h1 * fy;
}

// ---------------------------------------------------------------- Gaussian blur, row pass
#define SIFT_ROW_T 256
__global__ void __launch_bounds__(SIFT_ROW_T)
sift_blur_row_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols, SiftTaps taps, size_t fstride)
{
    __shared__ float s[SIFT_ROW_T + SIFT_MAX_TAPS];
    const int y = blockIdx.y, x0 = blockIdx.x * SIFT_ROW_T, h = taps.n / 2;
    src += blockIdx.z * fstride;
    dst += blockIdx.z * fstride;
    const float* row = src + (size_t)y * cols;
    for (int i = threadIdx.x; i < SIFT_ROW_T + 2 * h; i += SIFT_ROW_T) {
        const int x = x0 - h + i;
        s[i] = x < cols + h ? row[sift_reflect101(x, cols)] : 0.f;
    }
    __syncthreads();
    const int x = x0 + threadIdx.x;
    if (x >= cols) return;
    const float* w = s + threadIdx.x;
    float acc = taps.k[0] * w[0];
    if (x < (cols & ~3)) {
#pragma unroll 4
        for (int j = 1; j < taps.n; ++j) acc = __fmaf_rn(w[j], taps.k[j], acc);
    } else {
        for (int j = 1; j < taps.n; ++j) acc = acc + w[j] * taps.k[j];
    }
    dst[(size_t)y * cols + x] = acc;
}

// column pass: writes the Gaussian image and (when prev != nullptr) the DoG image  gauss - prev
__global__ void __launch_bounds__(256)
sift_blur_col_kernel(const float* __restrict__ tmp, float* __restrict__ gauss, const float* __restrict__ prev, float* __restrict__ dog,
                     int rows, int cols, SiftTaps taps, size_t fstride)
{
    const int x = blockIdx.x * 64 + (threadIdx.x & 63), y = blockIdx.y * 4 + (threadIdx.x >> 6);
    if (x >= cols || y >= rows) return;
    const size_t fo = blockIdx.z * fstride;
    tmp += fo; gauss += fo;
    if (dog) { prev += fo; dog += fo; }
    const int h = taps.n / 2;
    float d = taps.k[h] * tmp[(size_t)y * cols + x];
    const bool fused = x < (cols & ~7);
    for (int j = 1; j <= h; ++j) {
        const float a = tmp[(size_t)sift_reflect101(y - j, rows) * cols + x], b = tmp[(size_t)sift_reflect101(y + j, rows) * cols + x];
        d = fused ? __fmaf_rn(taps.k[h + j], a + b, d) : d + taps.k[h + j] * (a + b);
    }
    gauss[(size_t)y * cols + x] = d;
    if (dog) dog[(size_t)y * cols + x] = d - prev[(size_t)y * cols + x];
}

// resize(src, Size(cols / 2, rows / 2), INTER_NEAREST): sx = min(floor(x * (1 / (dcols / scols))), scols - 1)
__global__ void __launch_bounds__(256)
sift_halve_kernel(const float* __restrict__ src, int srows, int scols, float* __restrict__ dst, int drows, int dcols, double ifx, double ify,
                  size_t fstride)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    src += blockIdx.z * fstride;
    dst += blockIdx.z * fstride;
    if (x >= dcols) return;
    const double fy = y * ify, fx = x * ifx;
    int sy = (int)fy; sy -= (sy > fy); if (sy > srows - 1) sy = srows - 1;
    int sx = (int)fx; sx -= (sx > fx); if (sx > scols - 1) sx = scols - 1;
    dst[(size_t)y * dcols + x] = src[(size_t)sy * scols + sx];
}

// ---------------------------------------------------------------- extrema + sub-pixel refinement (adjustLocalExtrema)
struct SiftOctave {
    const float* dog[SIFT_LAYERS + 2];   // frame 0 of the chunk; frame f at + f * fstride
    int rows, cols, o;
    size_t fstride;
};

#define DET2(x, y, z, w) __fmaf_rn((x), (y), -((z) * (w)))

__device__ bool sift_adjust(const SiftOctave& O, size_t fo, int& layer, int& r, int& c, SiftCand& out)
{
    const float img_scale = 1.f / 255, deriv_scale = img_scale * 0.5f, second_deriv_scale = img_scale, cross_deriv_scale = img_scale * 0.25f;
    const int cols = O.cols, rows = O.rows;
    float xi = 0, xr = 0, xc = 0;
    int i = 0;
#define AT(im, rr, cc) ((im)[(size_t)(rr) * cols + (cc)])
    for (; i < SIFT_MAX_INTERP_STEPS; ++i) {
        const float *img = O.dog[layer] + fo, *prev = O.dog[layer - 1] + fo, *next = O.dog[layer + 1] + fo;
        const float b0 = (AT(img, r, c + 1) - AT(img, r, c - 1)) * deriv_scale, b1 = (AT(img, r + 1, c) - AT(img, r - 1, c)) * deriv_scale,
                    b2 = (AT(next, r, c) - AT(prev, r, c)) * deriv_scale;
        const float v2 = AT(img, r, c) * 2;
        const float dxx = (AT(img, r, c + 1) + AT(img, r, c - 1) - v2) * second_deriv_scale;
        const float dyy = (AT(img, r + 1, c) + AT(img, r - 1, c) - v2) * second_deriv_scale;
        const float dss = (AT(next, r, c) + AT(prev, r, c) - v2) * second_deriv_scale;
        const float dxy = (AT(img, r + 1, c + 1) - AT(img, r + 1, c - 1) - AT(img, r - 1, c + 1) + AT(img, r - 1, c - 1)) * cross_deriv_scale;
        const float dxs = (AT(next, r, c + 1) - AT(next, r, c - 1) - AT(prev, r, c + 1) + AT(prev, r, c - 1)) * cross_deriv_scale;
        const float dys = (AT(next, r + 1, c) - AT(next, r - 1, c) - AT(prev, r + 1, c) + AT(prev, r - 1, c)) * cross_deriv_scale;
        const float a00 = dxx, a01 = dxy, a02 = dxs, a10 = dxy, a11 = dyy, a12 = dys, a20 = dxs, a21 = dys, a22 = dss;
        float X0 = 0, X1 = 0, X2 = 0;
        {
            const float P = DET2(a11, a22, a21, a12), Q = DET2(a10, a22, a20, a12), Rr = DET2(a10, a21, a20, a11);
            float d = __fmaf_rn(a02, Rr, __fmaf_rn(a00, P, -(a01 * Q)));
            if (d != 0) {
                d = 1 / d;
                const float P0 = DET2(a11, a22, a12, a21), Q0 = DET2(b1, a22, a12, b2), R0 = DET2(b1, a21, a11, b2);
                const float Q1 = DET2(a10, a22, a12, a20), R1 = DET2(a10, b2, b1, a20);
                const float P2 = DET2(a11, b2, b1, a21), R2 = DET2(a10, a21, a11, a20);
                X0 = d * __fmaf_rn(a02, R0, __fmaf_rn(b0, P0, -(a01 * Q0)));
                X1 = d * __fmaf_rn(a02, R1, __fmaf_rn(a00, Q0, -(b0 * Q1)));
                X2 = d * __fmaf_rn(b0, R2, __fmaf_rn(a00, P2, -(a01 * R1)));
            }
        }
        xi = -X2; xr = -X1; xc = -X0;
        if (fabsf(xi) < 0.5f && fabsf(xr) < 0.5f && fabsf(xc) < 0.5f) break;
        if (fabsf(xi) > (float)(INT_MAX / 3) || fabsf(xr) > (float)(INT_MAX / 3) || fabsf(xc) > (float)(INT_MAX / 3)) return false;
        c += __float2int_rn(xc); r += __float2int_rn(xr); layer += __float2int_rn(xi);
        if (layer < 1 || layer > SIFT_LAYERS || c < SIFT_IMG_BORDER || c >= cols - SIFT_IMG_BORDER || r < SIFT_IMG_BORDER || r >= rows - SIFT_IMG_BORDER)
            return false;
    }
    if (i >= SIFT_MAX_INTERP_STEPS) return false;
    float contr;
    {
        const float *img = O.dog[layer] + fo, *prev = O.dog[layer - 1] + fo, *next = O.dog[layer + 1] + fo;
        const float b0 = (AT(img, r, c + 1) - AT(img, r, c - 1)) * deriv_scale, b1 = (AT(img, r + 1, c) - AT(img, r - 1, c)) * deriv_scale,
                    b2 = (AT(next, r, c) - AT(prev, r, c)) * deriv_scale;
        const float t = b0 * xc + b1 * xr + b2 * xi;
        contr = __fmaf_rn(AT(img, r, c), img_scale, t * 0.5f);
        if (fabsf(contr) * SIFT_LAYERS < 0.04f) return false;
        const float v2 = AT(img, r, c) * 2.f;
        const float dxx = (AT(img, r, c + 1) + AT(img, r, c - 1) - v2) * second_deriv_scale;
        const float dyy = (AT(img, r + 1, c) + AT(img, r - 1, c) - v2) * second_deriv_scale;
        const float dxy = (AT(img, r + 1, c + 1) - AT(img, r + 1, c - 1) - AT(img, r - 1, c + 1) + AT(img, r - 1, c - 1)) * cross_deriv_scale;
        const float tr = dxx + dyy, det = dxx * dyy - dxy * dxy;
        const float et = 10.f;
        if (det <= 0 || tr * tr * et >= (et + 1) * (et + 1) * det) return false;
    }
#undef AT
    const int octv = O.o;
    out.x = (c + xc) * (1 << octv);
    out.y = (r + xr) * (1 << octv);
    out.octave_code = octv + (layer << 8) + (__double2int_rn(((double)xi + 0.5) * 255) << 16);
    out.size = 1.6f * (float)exp2((double)((layer + xi) / SIFT_LAYERS)) * (1 << octv) * 2;
    out.response = fabsf(contr);
    out.o = octv; out.layer = layer; out.r = r; out.c = c;
    return true;
}

__global__ void __launch_bounds__(256)
sift_extrema_kernel(SiftOctave O, SiftCand* __restrict__ cands, int* __restrict__ n_cands, int cap)
{
    const int c = SIFT_IMG_BORDER + blockIdx.x * 64 + (threadIdx.x & 63), r = SIFT_IMG_BORDER + blockIdx.y * 4 + (threadIdx.x >> 6);
    const int f = blockIdx.z / SIFT_LAYERS, layer0 = 1 + blockIdx.z - f * SIFT_LAYERS;
    if (c >= O.cols - SIFT_IMG_BORDER || r >= O.rows - SIFT_IMG_BORDER) return;
    const int cols = O.cols;
    const float *img = O.dog[layer0] + f * O.fstride, *prev = O.dog[layer0 - 1] + f * O.fstride, *next = O.dog[layer0 + 1] + f * O.fstride;
    const float val = img[(size_t)r * cols + c];
    if (!(fabsf(val) > 1.f)) return;      // threshold = cvFloor(0.5 * 0.04 / 3 * 255) = 1
    bool ext = true;
    if (val > 0) {
#pragma unroll
        for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
            for (int dc = -1; dc <= 1; ++dc) {
                const size_t q = (size_t)(r + dr) * cols + (c + dc);
                ext = ext && val >= img[q] && val >= prev[q] && val >= next[q];
            }
    } else {
#pragma unroll
        for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
            for (int dc = -1; dc <= 1; ++dc) {
                const size_t q = (size_t)(r + dr) * cols + (c + dc);
                ext = ext && val <= img[q] && val <= prev[q] && val <= next[q];
            }
    }
    if (!ext) return;
    SiftCand cd;
    int layer = layer0, r1 = r, c1 = c;
    if (!sift_adjust(O, f * O.fstride, layer, r1, c1, cd)) return;
    cd.f = f;
    const int slot = atomicAdd(n_cands, 1);
    if (slot < cap) cands[slot] = cd;
}

// ---------------------------------------------------------------- orientation histograms: one CTA per extremum
__device__ __forceinline__ float sift_fast_atan2(float y, float x)
{
    const float scale = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale;
    const float p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
    const float ax = fabsf(x), ay = fabsf(y);
    const float c = fminf(ax, ay) / (fmaxf(ax, ay) + (float)DBL_EPSILON);
    const float cc = c * c;
    float a = __fmaf_rn(__fmaf_rn(__fmaf_rn(cc, p7, p5), cc, p3), cc, p1) * c;
    if (!(ax >= ay)) a = 90.f - a;
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

struct SiftPyrDev {
    const float* gauss[SIFT_MAX_OCTAVES][SIFT_LAYERS + 3];   // frame 0 of the chunk; frame f at + f * fstride
    int rows[SIFT_MAX_OCTAVES], cols[SIFT_MAX_OCTAVES];
    size_t fstride;
};

#define SIFT_ORI_T 128
__global__ void __launch_bounds__(SIFT_ORI_T)
sift_orientation_kernel(SiftPyrDev P, const SiftCand* __restrict__ cands, int n_cands, SiftKp* __restrict__ kps, int* __restrict__ n_kps, int cap)
{
    __shared__ signed char s_bin[SIFT_ORI_T];
    __shared__ float s_val[SIFT_ORI_T];
    __shared__ float s_hist[SIFT_ORI_BINS + 4];
    __shared__ float s_sm[SIFT_ORI_BINS];
    const int ci = blockIdx.x;
    if (ci >= n_cands) return;
    const SiftCand cd = cands[ci];
    const int o = cd.o, rows = P.rows[o], cols = P.cols[o], n = SIFT_ORI_BINS;
    const float* img = P.gauss[o][cd.layer] + cd.f * P.fstride;
    const float scl_octv = cd.size * 0.5f / (1 << o);
    const int radius = __float2int_rn(4.5f * scl_octv);
    const float sigma = 1.5f * scl_octv;
    const float expf_scale = -1.f / (2.f * sigma * sigma);
    const int side = 2 * radius + 1, total = side * side;
    float hist = 0.f;       // thread b < 36 owns bin b
    for (int base = 0; base < total; base += SIFT_ORI_T) {
        const int k = base + threadIdx.x;
        int bin = -1;
        float v = 0.f;
        if (k < total) {
            const int i = k / side - radius, j = k - (k / side) * side - radius;
            const int y = cd.r + i, x = cd.c + j;
            if (!(y <= 0 || y >= rows - 1 || x <= 0 || x >= cols - 1)) {
                const float dx = img[(size_t)y * cols + x + 1] - img[(size_t)y * cols + x - 1];
                const float dy = img[(size_t)(y - 1) * cols + x] - img[(size_t)(y + 1) * cols + x];
                const float w = sift_exp((float)(i * i + j * j) * expf_scale);
                const float ori = sift_fast_atan2(dy, dx);
                const float mag = sqrtf(dx * dx + dy * dy);
                bin = __float2int_rn((n / 360.f) * ori);
                if (bin >= n) bin -= n;
                if (bin < 0) bin += n;
                v = w * mag;
            }
        }
        s_bin[threadIdx.x] = (signed char)bin;
        s_val[threadIdx.x] = v;
        __syncthreads();
        if (threadIdx.x < n) {
            const int m = min(SIFT_ORI_T, total - base);
            for (int q = 0; q < m; ++q)
                if (s_bin[q] == (int)threadIdx.x) hist = hist + s_val[q];      // raster order, one owner per bin
        }
        __syncthreads();
    }
    if (threadIdx.x < n) s_hist[2 + threadIdx.x] = hist;
    __syncthreads();
    if (threadIdx.x == 0) { s_hist[1] = s_hist[2 + n - 1]; s_hist[0] = s_hist[2 + n - 2]; s_hist[2 + n] = s_hist[2]; s_hist[2 + n + 1] = s_hist[3]; }
    __syncthreads();
    if (threadIdx.x < n) {
        const float* t = s_hist + 2 + threadIdx.x;
        float hv;
        if (threadIdx.x < 32) hv = __fmaf_rn(t[-2] + t[2], 1.f / 16.f, __fmaf_rn(t[-1] + t[1], 4.f / 16.f, t[0] * (6.f / 16.f)));
        else hv = (t[-2] + t[2]) * (1.f / 16.f) + (t[-1] + t[1]) * (4.f / 16.f) + t[0] * (6.f / 16.f);
        s_sm[threadIdx.x] = hv;
    }
    __syncthreads();
    if (threadIdx.x < n) {
        float omax = s_sm[0];
        for (int q = 1; q < n; ++q) omax = fmaxf(omax, s_sm[q]);
        const float mag_thr = (float)(omax * 0.8f);
        const int j = threadIdx.x, l = j > 0 ? j - 1 : n - 1, r2 = j < n - 1 ? j + 1 : 0;
        const float hj = s_sm[j], hl = s_sm[l], hr = s_sm[r2];
        if (hj > hl && hj > hr && hj >= mag_thr) {
            float bin = j + 0.5f * (hl - hr) / (hl - 2 * hj + hr);
            bin = bin < 0 ? n + bin : bin >= n ? bin - n : bin;
            float angle = 360.f - (float)((360.f / n) * bin);
            if (fabsf(angle - 360.f) < FLT_EPSILON) angle = 0.f;
            const int slot = atomicAdd(n_kps, 1);
            if (slot < cap) {
                SiftKp kp;
                kp.x = cd.x; kp.y = cd.y; kp.size = cd.size; kp.angle = angle; kp.response = cd.response;
                kp.octave_code = cd.octave_code; kp.o = cd.o; kp.layer = cd.layer; kp.f = cd.f;
                kps[slot] = kp;
            }
        }
    }
}

// ---------------------------------------------------------------- descriptors: one CTA per keypoint
#define SIFT_DESC_T 128
#define SIFT_D 4
#define SIFT_N 8
#define SIFT_HIST ((SIFT_D + 2) * (SIFT_D + 2) * (SIFT_N + 2))

__global__ void __launch_bounds__(SIFT_DESC_T)
sift_descriptor_kernel(SiftPyrDev P, const SiftKp* __restrict__ kps, int n_kps, float* __restrict__ desc)
{   // kps: the ordered, deduplicated list with the freed slots marked f = -1; row ki of desc belongs to kps[ki]
    __shared__ float s_hist[SIFT_HIST];
    __shared__ float s_v[8][SIFT_DESC_T];
    __shared__ int s_cell[SIFT_DESC_T];        // ((r0 + 1) * 6 + (c0 + 1)) * 16 + o0 of the compacted valid samples, in raster order
    __shared__ int s_warp_cnt[SIFT_DESC_T / 32];
    __shared__ float s_raw[SIFT_D * SIFT_D * SIFT_N];
    __shared__ float s_scale[2];
    const int ki = blockIdx.x;
    if (ki >= n_kps) return;
    const SiftKp kp = kps[ki];
    if (kp.f < 0) return;
    const int d = SIFT_D, n = SIFT_N;
    // detectAndCompute: kpt.octave / pt / size are shifted by firstOctave = -1 before the descriptors; unpackOctave then scales
    // them back to the octave's own resolution.  In pyramid-index terms: scale = 1 / 2^o applied to the unshifted values,
    // but through cv2's own float operations: pt * 0.5, size * 0.5, then * scale with scale = 2 (o = 0) or 1 / 2^(o - 1).
    const int o = kp.o;
    const float scale = o == 0 ? 2.f : 1.f / (float)(1 << (o - 1));
    const float ptx = (kp.x * 0.5f) * scale, pty = (kp.y * 0.5f) * scale;
    const float size = (kp.size * 0.5f) * scale;
    float ori = 360.f - kp.angle;
    if (fabsf(ori - 360.f) < FLT_EPSILON) ori = 0.f;
    const float scl = size * 0.5f;
    const int rows = P.rows[o], cols = P.cols[o];
    const float* img = P.gauss[o][kp.layer] + kp.f * P.fstride;
    const int px = __float2int_rn(ptx), py = __float2int_rn(pty);
    float cos_t = (float)cos((double)(ori * (float)(3.14159265358979323846 / 180)));
    float sin_t = (float)sin((double)(ori * (float)(3.14159265358979323846 / 180)));
    const float bins_per_rad = n / 360.f;
    const float exp_scale = -1.f / (d * d * 0.5f);
    const float hist_width = 3.f * scl;
    int radius = __float2int_rn(hist_width * 1.4142135623730951f * (d + 1) * 0.5f);
    const int diag = (int)sqrt((double)cols * cols + (double)rows * rows);
    if (radius > diag) radius = diag;
    cos_t /= hist_width; sin_t /= hist_width;
    for (int q = threadIdx.x; q < SIFT_HIST; q += SIFT_DESC_T) s_hist[q] = 0.f;
    const int side = 2 * radius + 1;
    const long long total = (long long)side * side;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // owner of the histogram bins (cc, oo), all six rr: threads 0 .. 59
    const int own_cc = threadIdx.x / 10, own_oo = threadIdx.x - own_cc * 10;
    __syncthreads();
    for (long long base = 0; base < total; base += SIFT_DESC_T) {
        const long long k = base + threadIdx.x;
        bool valid = false;
        int cell = 0;
        float v[8];
        if (k < total) {
            const int i = (int)(k / side) - radius, j = (int)(k - (k / side) * side) - radius;
            const float c_rot = j * cos_t - i * sin_t;
            const float r_rot = j * sin_t + i * cos_t;
            float rbin = r_rot + d / 2 - 0.5f;
            float cbin = c_rot + d / 2 - 0.5f;
            const int r = py + i, c = px + j;
            if (rbin > -1 && rbin < d && cbin > -1 && cbin < d && r > 0 && r < rows - 1 && c > 0 && c < cols - 1) {
                valid = true;
                const float dx = img[(size_t)r * cols + c + 1] - img[(size_t)r * cols + c - 1];
                const float dy = img[(size_t)(r - 1) * cols + c] - img[(size_t)(r + 1) * cols + c];
                const float w = sift_exp((c_rot * c_rot + r_rot * r_rot) * exp_scale);
                const float ang = sift_fast_atan2(dy, dx);
                const float mag = sqrtf(dx * dx + dy * dy) * w;
                float obin = (ang - ori) * bins_per_rad;
                const int r0 = sift_floor(rbin), c0 = sift_floor(cbin);
                int o0 = sift_floor(obin);
                rbin -= r0; cbin -= c0; obin -= o0;
                if (o0 < 0) o0 += n;
                if (o0 >= n) o0 -= n;
                const float v_r1 = mag * rbin, v_r0 = mag - v_r1;
                const float v_rc11 = v_r1 * cbin, v_rc10 = v_r1 - v_rc11;
                const float v_rc01 = v_r0 * cbin, v_rc00 = v_r0 - v_rc01;
                const float v_rco111 = v_rc11 * obin, v_rco110 = v_rc11 - v_rco111;
                const float v_rco101 = v_rc10 * obin, v_rco100 = v_rc10 - v_rco101;
                const float v_rco011 = v_rc01 * obin, v_rco010 = v_rc01 - v_rco011;
                const float v_rco001 = v_rc00 * obin, v_rco000 = v_rc00 - v_rco001;
                // v[dr * 4 + dc * 2 + do]
                v[0] = v_rco000; v[1] = v_rco001; v[2] = v_rco010; v[3] = v_rco011;
                v[4] = v_rco100; v[5] = v_rco101; v[6] = v_rco110; v[7] = v_rco111;
                cell = ((r0 + 1) * 6 + (c0 + 1)) * 16 + o0;
            }
        }
        // order-preserving compaction of the valid samples of this chunk
        const unsigned bal = __ballot_sync(0xffffffffu, valid);
        if (lane == 0) s_warp_cnt[warp] = __popc(bal);
        __syncthreads();
        int off = __popc(bal & ((1u << lane) - 1));
        int m = 0;
        for (int w2 = 0; w2 < SIFT_DESC_T / 32; ++w2) { if (w2 < warp) off += s_warp_cnt[w2]; m += s_warp_cnt[w2]; }
        if (valid) {
            s_cell[off] = cell;
#pragma unroll
            for (int q = 0; q < 8; ++q) s_v[q][off] = v[q];
        }
        __syncthreads();
        if (threadIdx.x < 60) {
            for (int q = 0; q < m; ++q) {
                const int cl = s_cell[q];
                const int o0 = cl & 15, rc = cl >> 4, c1 = rc % 6, r1 = rc / 6;      // r1 = r0 + 1, c1 = c0 + 1
                const int dc = own_cc - c1, dO = own_oo - o0;
                if ((unsigned)dc <= 1u && (unsigned)dO <= 1u) {
                    float* hp = s_hist + ((r1 * 6 + own_cc) * 10 + own_oo);
                    hp[0] = hp[0] + s_v[dc * 2 + dO][q];
                    hp[60] = hp[60] + s_v[4 + dc * 2 + dO][q];
                }
            }
        }
        __syncthreads();
    }
    // circular orientation bins, copy out
    if (threadIdx.x < d * d * n) {
        const int k2 = threadIdx.x % n, j = (threadIdx.x / n) % d, i = threadIdx.x / (n * d);
        const int idx = ((i + 1) * (d + 2) + (j + 1)) * (n + 2);
        float hv = s_hist[idx + k2];
        if (k2 < 2) hv = hv + s_hist[idx + n + k2];
        s_raw[threadIdx.x] = hv;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int len = d * d * n;
        float nrm2 = 0;
        for (int k2 = 0; k2 < len; ++k2) nrm2 = nrm2 + s_raw[k2] * s_raw[k2];
        const float thr = sqrtf(nrm2) * 0.2f;
        nrm2 = 0;
        for (int k2 = 0; k2 < len; ++k2) { const float val = fminf(s_raw[k2], thr); nrm2 = nrm2 + val * val; }
        s_scale[0] = thr;
        s_scale[1] = 512.f / fmaxf(sqrtf(nrm2), FLT_EPSILON);
    }
    __syncthreads();
    if (threadIdx.x < d * d * n) {
        const float val = fminf(s_raw[threadIdx.x], s_scale[0]);
        int q = __float2int_rn(val * s_scale[1]);
        q = q < 0 ? 0 : q > 255 ? 255 : q;
        desc[(size_t)ki * 128 + threadIdx.x] = (float)q;
    }
}

// ---------------------------------------------------------------- cv2's keypoint order, duplicate removal
// KeyPointsFilter::removeDuplicatedSorted (features2d/src/keypoint.cpp) sorts by (x, y, -size, angle, -response, -octave) and
// drops every keypoint equal in (x, y, size, angle) to the one before it.  The frame comes first, so one sort orders every
// frame of a chunk.  Keypoints equal in all six fields are identical (descriptor included), so their order is immaterial.
struct SiftKpLess {
    __device__ __forceinline__ bool operator()(const SiftKp& a, const SiftKp& b) const
    {
        if (a.f != b.f) return a.f < b.f;
        if (a.x != b.x) return a.x < b.x;
        if (a.y != b.y) return a.y < b.y;
        if (a.size != b.size) return a.size > b.size;
        if (a.angle != b.angle) return a.angle < b.angle;
        if (a.response != b.response) return a.response > b.response;
        return a.octave_code > b.octave_code;
    }
};

#define SIFT_DEDUP_T 256
// One CTA per frame of the chunk: the frame's run [lo, hi) of the sorted list, first of each (x, y, size, angle) group kept in
// order (cta_compact) at out[lo + rank]; the rest of the run is marked free.  Writes the kept keypoints in the
// caller's format (firstOctave = -1 undone: coordinates and size halved, octave - 1 in the low byte) at kp6[base + lo + rank],
// and per frame the count and the first row.
// Detection mask (mask_off != nullptr): frame f's mask is at mask + mask_off[f] (rows `mask_pitch` bytes apart; < 0: none).
// A keypoint whose byte at ((int)(y + 0.5f), (int)(x + 0.5f)) of the halved coordinates is 0 is dropped as well, as cv2's
// KeyPointsFilter::runByPixelsMask drops it after the duplicates; duplicates share (x, y), so the two filters commute.
__global__ void __launch_bounds__(SIFT_DEDUP_T)
sift_dedup_kernel(const SiftKp* __restrict__ sorted, int n, SiftKp* __restrict__ out, float* __restrict__ kp6, int base,
                  int* __restrict__ n_frame, int* __restrict__ first_row, const uint8_t* __restrict__ mask,
                  const long long* __restrict__ mask_off, int mask_pitch)
{
    __shared__ int s_lo, s_hi;
    const int f = blockIdx.x;
    const uint8_t* fm = mask_off && mask_off[f] >= 0 ? mask + mask_off[f] : nullptr;
    if (threadIdx.x < 2) {   // lower bounds of f and f + 1
        const int key = f + threadIdx.x;
        int a = 0, b = n;
        while (a < b) { const int m = (a + b) >> 1; if (sorted[m].f < key) a = m + 1; else b = m; }
        if (threadIdx.x == 0) s_lo = a; else s_hi = a;
    }
    __syncthreads();
    const int lo = s_lo, hi = s_hi;
    const int cnt = cta_compact<SIFT_DEDUP_T>(hi - lo, [&](int j) {
        const SiftKp& k = sorted[lo + j];
        if (fm) {
            const int mx = (int)__fadd_rn(__fmul_rn(k.x, 0.5f), 0.5f), my = (int)__fadd_rn(__fmul_rn(k.y, 0.5f), 0.5f);
            if (!fm[(size_t)my * mask_pitch + mx]) return false;
        }
        if (j == 0) return true;
        const SiftKp& p = sorted[lo + j - 1];
        return p.x != k.x || p.y != k.y || p.size != k.size || p.angle != k.angle;
    }, [&](int j, int o) {
        const SiftKp k = sorted[lo + j];
        out[lo + o] = k;
        const int oc = (k.octave_code & ~255) | ((k.octave_code - 1) & 255);
        float* q = kp6 + (size_t)(base + lo + o) * 6;
        q[0] = k.x * 0.5f; q[1] = k.y * 0.5f; q[2] = k.size * 0.5f; q[3] = k.angle; q[4] = k.response;
        memcpy(&q[5], &oc, 4);
    });
    for (int i = lo + cnt + threadIdx.x; i < hi; i += SIFT_DEDUP_T) out[i].f = -1;
    if (threadIdx.x == 0) { n_frame[f] = cnt; first_row[f] = base + lo; }
}

// ---------------------------------------------------------------- host
static int sift_kernel_taps(double sigma, SiftTaps* t)
{
    // cv::getGaussianKernel(n, sigma, CV_32F): x doubled, scale -0.125 / sigma^2, normalised in double, cast to float
    const int n = (int)lrint(sigma * 4 * 2 + 1) | 1;
    if (n > SIFT_MAX_TAPS) return -1;
    const double scale2x = -0.125 / (sigma * sigma);
    const int n2 = (n - 1) / 2;
    double vals[SIFT_MAX_TAPS];
    double sum = 0;
    for (int i = 0, x = 1 - n; i < n2; ++i, x += 2) { vals[i] = exp((double)(x * x) * scale2x); sum += vals[i]; }
    sum *= 2; sum += 1.0;
    const double mul1 = 1.0 / sum;
    for (int i = 0; i < n2; ++i) { const float v = (float)(vals[i] * mul1); t->k[i] = v; t->k[n - 1 - i] = v; }
    t->k[n2] = (float)(1.0 * mul1);
    for (int i = n; i < SIFT_MAX_TAPS; ++i) t->k[i] = 0.f;
    t->n = n;
    return 0;
}

static int sift_blur(b200vo_ctx* ctx, const float* src, float* tmp, float* gauss, const float* prev, float* dog, int rows, int cols, double sigma,
                     int nf, size_t fstride)
{
    SiftTaps t;
    if (sift_kernel_taps(sigma, &t)) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "Gaussian kernel of sigma %g needs more than %d taps", sigma, SIFT_MAX_TAPS);
    sift_blur_row_kernel<<<dim3((cols + SIFT_ROW_T - 1) / SIFT_ROW_T, rows, nf), SIFT_ROW_T, 0, ctx->stream>>>(src, tmp, rows, cols, t, fstride);
    sift_blur_col_kernel<<<dim3((cols + 63) / 64, (rows + 3) / 4, nf), 256, 0, ctx->stream>>>(tmp, gauss, prev, dog, rows, cols, t, fstride);
    ctx->launches += 2;
    return 0;
}

// Scale space of one frame: the doubled image, the row-pass scratch and per octave 6 Gaussian + 5 DoG images.  Octaves whose
// images have fewer than 11 rows or columns cannot hold an extremum (5-pixel border) and are not built.
struct SiftGeom {
    int brows, bcols, n_act;
    int orows[SIFT_MAX_OCTAVES], ocols[SIFT_MAX_OCTAVES];
    size_t o_up, o_tmp, o_g[SIFT_MAX_OCTAVES][SIFT_LAYERS + 3], o_d[SIFT_MAX_OCTAVES][SIFT_LAYERS + 2];
    size_t frame_bytes;
};

static void sift_geom(int rows, int cols, SiftGeom& G)
{
    G.brows = rows * 2; G.bcols = cols * 2;
    const int mn = G.bcols < G.brows ? G.bcols : G.brows;
    int n_oct = (int)lrint(log((double)mn) / log(2.) - 2) + 1;       // firstOctave = -1
    if (n_oct < 1) n_oct = 1;
    G.n_act = 0;
    for (int o = 0, r = G.brows, c = G.bcols; o < n_oct && o < SIFT_MAX_OCTAVES; ++o, r /= 2, c /= 2) {
        if (r < 2 * SIFT_IMG_BORDER + 1 || c < 2 * SIFT_IMG_BORDER + 1) break;
        G.orows[o] = r; G.ocols[o] = c; G.n_act = o + 1;
    }
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o2 = off; off += vo_align(bytes, 256); return o2; };
    const size_t base_px = (size_t)G.brows * G.bcols;
    G.o_up = take(base_px * 4); G.o_tmp = take(base_px * 4);
    for (int o = 0; o < G.n_act; ++o) {
        const size_t px = (size_t)G.orows[o] * G.ocols[o];
        for (int i = 0; i < SIFT_LAYERS + 3; ++i) G.o_g[o][i] = take(px * 4);
        for (int i = 0; i < SIFT_LAYERS + 2; ++i) G.o_d[o][i] = take(px * 4);
    }
    G.frame_bytes = off;
}

#define SIFT_CAND_CAP (1 << 18)    // extrema per frame
#define SIFT_KP_CAP (1 << 18)      // keypoints per frame
// The workspace of one chunk of frames, with the quarter vo_reserve adds, fits this budget (about 150 MB per KITTI-sized
// frame with its extrema and keypoints: 21 frames).
#define SIFT_CHUNK_BYTES ((size_t)4 << 30)

static size_t sift_per_frame_bytes(const SiftGeom& G)
{
    return G.frame_bytes + (size_t)SIFT_CAND_CAP * sizeof(SiftCand) + (size_t)2 * SIFT_KP_CAP * sizeof(SiftKp);
}

// grows b to `bytes`, keeping its first `used` bytes
static int sift_reserve_keep(b200vo_ctx* ctx, DevBuf& b, size_t used, size_t bytes)
{
    if (bytes <= b.cap) return 0;
    DevBuf nb;
    VO_TRY(vo_reserve(ctx, nb, bytes));
    if (used) VO_CUDA(ctx, cudaMemcpyAsync(nb.p, b.p, used, cudaMemcpyDeviceToDevice, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (b.p) VO_CUDA(ctx, cudaFree(b.p));
    b = nb;
    return 0;
}

int vo_sift_frames(b200vo_ctx* ctx, const uint8_t* d_raw, size_t raw_stride, int n_frames, int rows, int cols, bool want_desc,
                   int* d_n_frame, int* d_first_row, int* n_rows, int row0, size_t row_stride, const uint8_t* d_mask,
                   const long long* d_mask_off)
{
    const int L = SIFT_LAYERS;
    if (!row_stride) row_stride = (size_t)cols;
    SiftGeom G;
    sift_geom(rows, cols, G);
    const size_t per_frame = sift_per_frame_bytes(G);
    const int chunk = (int)std::max<size_t>(1, SIFT_CHUNK_BYTES / 5 * 4 / per_frame);
    double sig[SIFT_LAYERS + 3];
    sig[0] = 1.6;
    const double kk = pow(2., 1. / L);
    for (int i = 1; i < L + 3; ++i) {
        const double sp = pow(kk, (double)(i - 1)) * 1.6, st = sp * kk;
        sig[i] = sqrt(st * st - sp * sp);
    }
    const float sg = 1.6f;
    const float sig_diff = sqrtf(std::max(sg * sg - 0.5f * 0.5f * 4, 0.01f));     // createInitialImage: float arithmetic
    const size_t fs = G.frame_bytes / 4;   // frame stride of the workspace, in floats
    int base = row0;                       // output rows written so far
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = std::min(chunk, n_frames - f0);
        const size_t cand_cap = (size_t)nf * SIFT_CAND_CAP, kp_cap = (size_t)nf * SIFT_KP_CAP;
        const size_t o_cand = vo_align((size_t)nf * G.frame_bytes, 256), o_kp = o_cand + vo_align(cand_cap * sizeof(SiftCand), 256);
        const size_t o_sorted = o_kp + vo_align(kp_cap * sizeof(SiftKp), 256), o_cnt = o_sorted + vo_align(kp_cap * sizeof(SiftKp), 256);
        VO_TRY(vo_reserve(ctx, ctx->d_sift, o_cnt + 256));
        uint8_t* ws = (uint8_t*)ctx->d_sift.p;
        int* d_cnt = (int*)(ws + o_cnt);
        VO_CUDA(ctx, cudaMemsetAsync(d_cnt, 0, 8, ctx->stream));
        float* up = (float*)(ws + G.o_up);
        float* tmp = (float*)(ws + G.o_tmp);
        sift_upscale_kernel<<<dim3((G.bcols + 255) / 256, G.brows, nf), 256, 0, ctx->stream>>>(d_raw + (size_t)f0 * raw_stride, rows, cols,
                                                                                              row_stride, raw_stride, up, fs);
        ctx->launches++;
        SiftPyrDev P{};
        P.fstride = fs;
        for (int o = 0; o < G.n_act; ++o) {
            P.rows[o] = G.orows[o]; P.cols[o] = G.ocols[o];
            for (int i = 0; i < L + 3; ++i) P.gauss[o][i] = (const float*)(ws + G.o_g[o][i]);
        }
        for (int o = 0; o < G.n_act; ++o) {
            float* g0 = (float*)(ws + G.o_g[o][0]);
            if (o == 0) {
                VO_TRY(sift_blur(ctx, up, tmp, g0, nullptr, nullptr, G.brows, G.bcols, (double)sig_diff, nf, fs));
            } else {
                const double ifx = 1.0 / ((double)G.ocols[o] / G.ocols[o - 1]), ify = 1.0 / ((double)G.orows[o] / G.orows[o - 1]);
                sift_halve_kernel<<<dim3((G.ocols[o] + 255) / 256, G.orows[o], nf), 256, 0, ctx->stream>>>(
                    (const float*)(ws + G.o_g[o - 1][L]), G.orows[o - 1], G.ocols[o - 1], g0, G.orows[o], G.ocols[o], ifx, ify, fs);
                ctx->launches++;
            }
            for (int i = 1; i < L + 3; ++i)
                VO_TRY(sift_blur(ctx, (const float*)(ws + G.o_g[o][i - 1]), tmp, (float*)(ws + G.o_g[o][i]), (const float*)(ws + G.o_g[o][i - 1]),
                                 (float*)(ws + G.o_d[o][i - 1]), G.orows[o], G.ocols[o], sig[i], nf, fs));
            SiftOctave O{};
            for (int i = 0; i < L + 2; ++i) O.dog[i] = (const float*)(ws + G.o_d[o][i]);
            O.rows = G.orows[o]; O.cols = G.ocols[o]; O.o = o; O.fstride = fs;
            const int ew = G.ocols[o] - 2 * SIFT_IMG_BORDER, eh = G.orows[o] - 2 * SIFT_IMG_BORDER;
            sift_extrema_kernel<<<dim3((ew + 63) / 64, (eh + 3) / 4, nf * L), 256, 0, ctx->stream>>>(O, (SiftCand*)(ws + o_cand), d_cnt,
                                                                                                    (int)cand_cap);
            ctx->launches++;
        }
        VO_CUDA(ctx, cudaGetLastError());
        VO_TRY(vo_reserve_pinned(ctx, 256));
        int* h_cnt = (int*)ctx->h_pin;
        VO_CUDA(ctx, cudaMemcpyAsync(h_cnt, d_cnt, 4, cudaMemcpyDeviceToHost, ctx->stream));
        VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const int n_cand = h_cnt[0];
        if ((size_t)n_cand > cand_cap) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "%d scale-space extrema exceed the limit of %zu", n_cand, cand_cap);
        int n_kp = 0;
        if (n_cand > 0) {
            sift_orientation_kernel<<<n_cand, SIFT_ORI_T, 0, ctx->stream>>>(P, (const SiftCand*)(ws + o_cand), n_cand, (SiftKp*)(ws + o_kp), d_cnt + 1,
                                                                           (int)kp_cap);
            ctx->launches++;
            VO_CUDA(ctx, cudaGetLastError());
            VO_CUDA(ctx, cudaMemcpyAsync(h_cnt + 1, d_cnt + 1, 4, cudaMemcpyDeviceToHost, ctx->stream));
            VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            n_kp = h_cnt[1];
            if ((size_t)n_kp > kp_cap) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "%d keypoints exceed the limit of %zu", n_kp, kp_cap);
        }
        SiftKp* kps = (SiftKp*)(ws + o_kp);
        SiftKp* sorted = (SiftKp*)(ws + o_sorted);
        VO_TRY(sift_reserve_keep(ctx, ctx->d_sift_out[0], (size_t)base * 24, (size_t)(base + n_kp) * 24 + 256));
        if (want_desc) VO_TRY(sift_reserve_keep(ctx, ctx->d_sift_out[1], (size_t)base * 512, (size_t)(base + n_kp) * 512 + 256));
        if (n_kp > 0) {
            size_t tb = 0;
            VO_CUDA(ctx, cub::DeviceMergeSort::SortKeysCopy(nullptr, tb, kps, sorted, n_kp, SiftKpLess(), ctx->stream));
            VO_TRY(vo_reserve(ctx, ctx->d_sift_sort, tb));
            VO_CUDA(ctx, cub::DeviceMergeSort::SortKeysCopy(ctx->d_sift_sort.p, tb, kps, sorted, n_kp, SiftKpLess(), ctx->stream));
            // CUB's merge sort: one block-sort launch, then a partition and a merge launch per pass over the tiles
            const int tile = cub::detail::merge_sort::policy_hub<SiftKp*>::MaxPolicy::MergeSortPolicy::ITEMS_PER_TILE;
            int passes = 0;
            for (int t = 1; t < (n_kp + tile - 1) / tile; t *= 2) ++passes;
            ctx->launches += 1 + 2 * passes;
        }
        sift_dedup_kernel<<<nf, SIFT_DEDUP_T, 0, ctx->stream>>>(sorted, n_kp, kps, (float*)ctx->d_sift_out[0].p, base, d_n_frame + f0,
                                                              d_first_row + f0, d_mask, d_mask_off ? d_mask_off + f0 : nullptr,
                                                              (int)row_stride);
        ctx->launches++;
        if (n_kp > 0 && want_desc) {
            sift_descriptor_kernel<<<n_kp, SIFT_DESC_T, 0, ctx->stream>>>(P, kps, n_kp, (float*)ctx->d_sift_out[1].p + (size_t)base * 128);
            ctx->launches++;
        }
        VO_CUDA(ctx, cudaGetLastError());
        base += n_kp;
    }
    *n_rows = base;
    return 0;
}

// the host forms of SIFT detectAndCompute; mask: uint8 rows x cols, `mask_step` bytes a row, or nullptr
static int sift_host(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols, size_t step, const uint8_t* mask, size_t mask_step,
                     int max_kp, float* kps_out, float* desc_out, int32_t* n_out)
{
    if (!ctx || !img || !n_out || rows <= 0 || cols <= 0 || step < (size_t)cols || max_kp < 0 || (max_kp > 0 && !kps_out) ||
        (mask && mask_step < (size_t)cols))
        return B200VO_E_BADARG;
    *n_out = 0;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    // upload (tight rows)
    VO_TRY(vo_reserve(ctx, ctx->d_stage_img[0], (size_t)rows * cols + 256));
    uint8_t* raw = (uint8_t*)ctx->d_stage_img[0].p;
    int* d_small = (int*)(raw + vo_align((size_t)rows * cols, 128));   // count | first row
    VO_CUDA(ctx, cudaMemcpy2DAsync(raw, cols, img, step, cols, rows, cudaMemcpyHostToDevice, ctx->stream));
    // the mask (tight rows, as the frame) after the one-entry table of its offset
    const long long* d_moff = nullptr;
    const uint8_t* d_mask = nullptr;
    if (mask) {
        VO_TRY(vo_reserve(ctx, ctx->d_mask, 256 + (size_t)rows * cols));
        const long long zero = 0;
        d_moff = (const long long*)ctx->d_mask.p;
        d_mask = (const uint8_t*)ctx->d_mask.p + 256;
        VO_CUDA(ctx, cudaMemcpyAsync(ctx->d_mask.p, &zero, sizeof(zero), cudaMemcpyHostToDevice, ctx->stream));
        VO_CUDA(ctx, cudaMemcpy2DAsync((uint8_t*)ctx->d_mask.p + 256, cols, mask, mask_step, cols, rows, cudaMemcpyHostToDevice, ctx->stream));
    }
    int n_rows = 0;
    VO_TRY(vo_sift_frames(ctx, raw, (size_t)rows * cols, 1, rows, cols, desc_out != nullptr, d_small, d_small + 1, &n_rows, 0, 0, d_mask,
                          d_moff));
    // rows [0, count) of the outputs are the keypoints in cv2's order
    const size_t b_k = vo_align((size_t)n_rows * 24, 256), b_d = desc_out ? (size_t)n_rows * 512 : 0;
    VO_TRY(vo_reserve_pinned(ctx, 256 + b_k + b_d));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    VO_CUDA(ctx, cudaMemcpyAsync(hp, d_small, 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_rows > 0) {
        VO_CUDA(ctx, cudaMemcpyAsync(hp + 256, ctx->d_sift_out[0].p, (size_t)n_rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
        if (desc_out) VO_CUDA(ctx, cudaMemcpyAsync(hp + 256 + b_k, ctx->d_sift_out[1].p, b_d, cudaMemcpyDeviceToHost, ctx->stream));
    }
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    const int cnt = *(const int*)hp;
    const int n_w = cnt < max_kp ? cnt : max_kp;
    if (n_w > 0) {
        memcpy(kps_out, hp + 256, (size_t)n_w * 24);
        if (desc_out) memcpy(desc_out, hp + 256 + b_k, (size_t)n_w * 512);
    }
    *n_out = cnt;
    return 0;
}

extern "C" int b200vo_sift_detect_and_compute(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols, size_t step, int max_kp,
                                              float* kps_out, float* desc_out, int32_t* n_out)
{
    return sift_host(ctx, img, rows, cols, step, nullptr, 0, max_kp, kps_out, desc_out, n_out);
}

extern "C" int b200vo_sift_detect_and_compute_masked(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols, size_t step,
                                                     const uint8_t* mask, size_t mask_step, int max_kp, float* kps_out,
                                                     float* desc_out, int32_t* n_out)
{
    return sift_host(ctx, img, rows, cols, step, mask, mask_step, max_kp, kps_out, desc_out, n_out);
}
