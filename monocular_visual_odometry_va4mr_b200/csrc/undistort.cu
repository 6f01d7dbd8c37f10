// Lens distortion removal as cv2 computes it: the fixed-point map of cv2.initUndistortRectifyMap(K, dist, None, Knew, size,
// CV_16SC2) (pinhole) or cv2.fisheye.initUndistortRectifyMap(K, D, I, Knew, size, CV_16SC2) (fisheye), and cv2.remap
// (INTER_LINEAR, BORDER_CONSTANT 0) through it.  K is the raw camera the coefficients belong to, Knew the camera of the
// undistorted image.  The map is evaluated in plain double (the build disables FMA contraction) and rounded to 1/32 px,
// which is what cv2's striped evaluation gives; the pyramid builder gathers level 0 through the same map (pyramid.cu).
#include <cmath>
#include <climits>
#include "internal.cuh"

bool vo_dist_valid(const double d[8])
{
    for (int i = 0; i < 8; ++i) if (!std::isfinite(d[i])) return false;
    return true;
}

// cvRound(a * 32) as x86 computes it: NaN, +-inf and values outside int32 become INT_MIN (so the pixel maps outside the image)
__device__ __forceinline__ int undist_round32(double a)
{
    a = a * 32.0;
    return (a > -2147483648.5 && a < 2147483647.5) ? __double2int_rn(a) : INT_MIN;
}

__device__ __forceinline__ short undist_sat16(int v) { return (short)max(-32768, min(32767, v)); }

// one thread per map entry of image blockIdx.y (the grid covers max_rows x max_cols, each image its own size); par row
// ([VO_LENS_PAR] doubles): raw fx, fy, cx, cy, new fx, fy, cx, cy, 8 coefficients, cols, rows.  A pixel is normalised by
// the new camera, distorted and projected with the raw one.  Pinhole: k1, k2, p1, p2, k3, k4, k5, k6, the source pixel
// saturated to int16 as cv2 stores it.  Fisheye: k1 .. k4, the source pixel wrapped modulo 2^16 as cv2.fisheye stores it.
template <int MODEL>
__global__ void __launch_bounds__(256)
undistort_map_kernel(const double* __restrict__ par, const int* __restrict__ im_of, int max_cols, int max_rows, short2* __restrict__ xy,
                     uint16_t* __restrict__ fr, size_t stride, int pitch)
{
    const double* q = par + VO_LENS_PAR * blockIdx.y;
    const int w = (int)q[16], h = (int)q[17];
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int i = (int)(p / max_cols), j = (int)(p - (long long)i * max_cols);
    if (i >= max_rows || i >= h || j >= w) return;
    const double fx = q[0], fy = q[1], cx = q[2], cy = q[3];
    const double x = (j - q[6]) / q[4], y = (i - q[7]) / q[5];
    double u, v;
    if (MODEL == B200VO_LENS_FISHEYE) {
        const double r = sqrt(x * x + y * y);
        const double th = atan(r);
        const double th2 = th * th, th4 = th2 * th2, th6 = th4 * th2, th8 = th4 * th4;
        const double thd = th * (1 + q[8] * th2 + q[9] * th4 + q[10] * th6 + q[11] * th8);
        const double s = r == 0 ? 1.0 : thd / r;
        u = fx * x * s + cx;
        v = fy * y * s + cy;
    } else {
        const double k1 = q[8], k2 = q[9], p1 = q[10], p2 = q[11], k3 = q[12], k4 = q[13], k5 = q[14], k6 = q[15];
        const double r2 = x * x + y * y;
        const double kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2);
        u = fx * (x * kr + p1 * 2 * x * y + p2 * (r2 + 2 * x * x)) + cx;
        v = fy * (y * kr + p1 * (r2 + 2 * y * y) + p2 * 2 * x * y) + cy;
    }
    const int iu = undist_round32(u), iv = undist_round32(v);
    const size_t o = (size_t)(im_of ? im_of[blockIdx.y] : blockIdx.y) * stride + (size_t)i * pitch + j;
    xy[o] = MODEL == B200VO_LENS_FISHEYE ? make_short2((short)(iu >> 5), (short)(iv >> 5))
                                         : make_short2(undist_sat16(iu >> 5), undist_sat16(iv >> 5));
    fr[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
}

void vo_lens_row(double row[VO_LENS_PAR], const VoIntrinsics& raw, const VoIntrinsics& cam, const double d[8], int cols, int rows)
{
    const double r[VO_LENS_PAR] = {raw.fx, raw.fy, raw.cx, raw.cy, cam.fx, cam.fy, cam.cx, cam.cy,
                                   d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7], (double)cols, (double)rows};
    memcpy(row, r, sizeof(r));
}

int vo_undistort_maps(b200vo_ctx* ctx, int model, const double* d_par, const int* d_im_of, int n, int max_rows, int max_cols,
                      short2* xy, uint16_t* fr, size_t stride, int pitch, cudaStream_t stream)
{
    const long long px = (long long)max_rows * max_cols;
    const dim3 grid((unsigned)((px + 255) / 256), n);
    if (model == B200VO_LENS_FISHEYE)
        undistort_map_kernel<B200VO_LENS_FISHEYE><<<grid, 256, 0, stream>>>(d_par, d_im_of, max_cols, max_rows, xy, fr, stride, pitch);
    else
        undistort_map_kernel<B200VO_LENS_PINHOLE><<<grid, 256, 0, stream>>>(d_par, d_im_of, max_cols, max_rows, xy, fr, stride, pitch);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// one thread = 4 consecutive pixels of frame blockIdx.z
__global__ void __launch_bounds__(256)
undistort_frames_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, size_t stride, size_t row, int w, int h,
                        VoUndist ud, const int* __restrict__ seq_of, int seq_shift, const VoSeqExt* __restrict__ ext)
{
    const int z = blockIdx.z;
    const int im = seq_of ? seq_of[z >> seq_shift] : z;
    if (ext) { w = ext[im].w[0]; h = ext[im].h[0]; }
    const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x0 >= w || y >= h) return;
    const uint8_t* s = src + z * stride;
    uint8_t* d = dst + z * stride + (size_t)y * row;
    const bool on = !ud.on || ud.on[im];
    const short2* xy = ud.xy + im * ud.stride;
    const uint16_t* fr = ud.fr + im * ud.stride;
    for (int x = x0; x < min(x0 + 4, w); ++x)
        d[x] = on ? (uint8_t)vo_undist_px(s, row, w, h, xy, fr, ud.pitch, x, y) : s[(size_t)y * row + x];
}

int vo_undistort_frames(b200vo_ctx* ctx, const uint8_t* src, uint8_t* dst, size_t stride, size_t row, int n, int rows, int cols,
                        const VoUndist& ud, const int* seq_of, int seq_shift, const VoSeqExt* ext, cudaStream_t stream)
{
    undistort_frames_kernel<<<dim3((cols + 1023) / 1024, rows, n), 256, 0, stream>>>(src, dst, stride, row, cols, rows, ud, seq_of,
                                                                                     seq_shift, ext);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// The one-call forms: src through the map of (model, K, d8, Knew) into dst, both rows x cols (inputs checked by the caller)
static int undistort_one(b200vo_ctx* ctx, int model, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                         const double d8[8], const double Knew[9], uint8_t* dst)
{
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t npx = (size_t)rows * cols;
    const size_t b_par = 256, b_xy = vo_align(npx * 4, 256), b_fr = vo_align(npx * 2, 256), b_img = vo_align(npx, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_undist, b_par + b_xy + b_fr + 2 * b_img));
    uint8_t* p = (uint8_t*)ctx->d_undist.p;
    double* d_par = (double*)p;
    short2* xy = (short2*)(p + b_par);
    uint16_t* fr = (uint16_t*)(p + b_par + b_xy);
    uint8_t* d_src = p + b_par + b_xy + b_fr;
    uint8_t* d_dst = d_src + b_img;
    VoIntrinsics raw, cam;
    vo_intrinsics_row(raw, K, VO_BOOT_EMAT_THR);
    vo_intrinsics_row(cam, Knew, VO_BOOT_EMAT_THR);
    double par[VO_LENS_PAR];
    vo_lens_row(par, raw, cam, d8, cols, rows);
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, st));
    VO_CUDA(ctx, cudaMemcpyAsync(d_par, par, sizeof(par), cudaMemcpyHostToDevice, st));
    VO_CUDA(ctx, cudaMemcpy2DAsync(d_src, (size_t)cols, src, step, (size_t)cols, (size_t)rows, cudaMemcpyHostToDevice, st));
    VO_TRY(vo_undistort_maps(ctx, model, d_par, nullptr, 1, rows, cols, xy, fr, npx, cols, st));
    VoUndist ud;
    ud.xy = xy; ud.fr = fr; ud.stride = npx; ud.pitch = cols;
    VO_TRY(vo_undistort_frames(ctx, d_src, d_dst, npx, (size_t)cols, 1, rows, cols, ud, nullptr, 0, nullptr, st));
    VO_CUDA(ctx, cudaMemcpyAsync(dst, d_dst, npx, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, st));
    VO_CUDA(ctx, cudaStreamSynchronize(st));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    return 0;
}

extern "C" int b200vo_undistort_new_camera(b200vo_ctx* ctx, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                                           const double* dist, int n_dist, const double Knew[9], uint8_t* dst)
{
    if (!ctx) return B200VO_E_BADARG;
    if (!src || !K || !Knew || !dst || (n_dist > 0 && !dist)) return vo_set_err(ctx, B200VO_E_BADARG, "null array");
    if (rows < 1 || cols < 1 || step < (size_t)cols) return vo_set_err(ctx, B200VO_E_BADARG, "bad image size or step");
    if (n_dist != 4 && n_dist != 5 && n_dist != 8) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "n_dist = %d: only 4, 5 or 8 coefficients", n_dist);
    if (!vo_intrinsics_valid(K)) return vo_set_err(ctx, B200VO_E_BADARG, "K is not a pinhole camera matrix");
    if (!vo_intrinsics_valid(Knew)) return vo_set_err(ctx, B200VO_E_BADARG, "Knew is not a pinhole camera matrix");
    double d8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n_dist; ++i) d8[i] = dist[i];
    if (!vo_dist_valid(d8)) return vo_set_err(ctx, B200VO_E_BADARG, "non-finite distortion coefficient");
    return undistort_one(ctx, B200VO_LENS_PINHOLE, src, rows, cols, step, K, d8, Knew, dst);
}

extern "C" int b200vo_undistort(b200vo_ctx* ctx, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                                const double* dist, int n_dist, uint8_t* dst)
{
    return b200vo_undistort_new_camera(ctx, src, rows, cols, step, K, dist, n_dist, K, dst);
}

extern "C" int b200vo_fisheye_undistort(b200vo_ctx* ctx, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                                        const double D[4], const double* Knew, uint8_t* dst)
{
    static const double eye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    if (!ctx) return B200VO_E_BADARG;
    if (!src || !K || !D || !dst) return vo_set_err(ctx, B200VO_E_BADARG, "null array");
    if (rows < 1 || cols < 1 || step < (size_t)cols) return vo_set_err(ctx, B200VO_E_BADARG, "bad image size or step");
    if (!Knew) Knew = eye;
    if (!vo_intrinsics_valid(K)) return vo_set_err(ctx, B200VO_E_BADARG, "K is not a pinhole camera matrix");
    if (!vo_intrinsics_valid(Knew)) return vo_set_err(ctx, B200VO_E_BADARG, "Knew is not a pinhole camera matrix");
    const double d8[8] = {D[0], D[1], D[2], D[3], 0, 0, 0, 0};
    if (!vo_dist_valid(d8)) return vo_set_err(ctx, B200VO_E_BADARG, "non-finite distortion coefficient");
    return undistort_one(ctx, B200VO_LENS_FISHEYE, src, rows, cols, step, K, d8, Knew, dst);
}
