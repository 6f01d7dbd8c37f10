/* The maps of the lens models whose undistorted camera Knew may differ from the raw camera K (test-only CPU oracle), in
 * cv2's fixed-point CV_16SC2 + CV_16UC1 layout (int16 source pixel, fraction (v & 31) * 32 + (u & 31)), evaluated per
 * pixel in plain double; orc_remap_linear (undistort_oracle.c) applies them.
 *   orc_undistort_map_new_camera: cv2.initUndistortRectifyMap(K, d, None, Knew, (cols, rows), CV_16SC2) -- the pinhole
 *          model of orc_undistort_map with x, y normalised by Knew and projected with K; the source pixel saturates.
 *   orc_fisheye_map: cv2.fisheye.initUndistortRectifyMap(K, D, I, Knew, (cols, rows), CV_16SC2) -- the equidistant model,
 *          theta_d = theta (1 + k1 theta^2 + k2 theta^4 + k3 theta^6 + k4 theta^8), theta = atan(r); the source pixel
 *          WRAPS modulo 2^16 ((short)(iu >> 5)), as cv2 stores it.
 * cv2 inverts Knew and accumulates the normalised coordinates along a row; the closed form (j - cx') / fx' gives the same
 * entries (tests/test_oracle_fisheye.py).
 * This file stands beside undistort_oracle.c rather than inside it so that the already pinned orc_undistort_map stays
 * byte for byte the code its tests validated: the pinhole expression and the rounding helpers are restated here (a second,
 * independently pinned copy), not shared.  test_oracle_fisheye.py checks that the two pinhole maps agree when Knew = K. */
#include <math.h>
#include <limits.h>
#include <stddef.h>
#include <stdint.h>

/* cvRound on x86 (cvtsd2si): NaN, +-inf and values outside int32 give INT_MIN */
static int lens_round(double a)
{
    if (!(a > -2147483648.5 && a < 2147483647.5)) return INT_MIN;
    return (int)rint(a);
}

static int16_t lens_sat16(int v) { return (int16_t)(v < -32768 ? -32768 : v > 32767 ? 32767 : v); }

void orc_undistort_map_new_camera(int rows, int cols, const double K[9], const double d[8], const double Knew[9], int16_t* xy,
                                  uint16_t* fr)
{
    const double fx = K[0], fy = K[4], cx = K[2], cy = K[5];
    const double nfx = Knew[0], nfy = Knew[4], ncx = Knew[2], ncy = Knew[5];
    const double k1 = d[0], k2 = d[1], p1 = d[2], p2 = d[3], k3 = d[4], k4 = d[5], k5 = d[6], k6 = d[7];
    for (int i = 0; i < rows; ++i)
        for (int j = 0; j < cols; ++j) {
            const double x = (j - ncx) / nfx, y = (i - ncy) / nfy;
            const double r2 = x * x + y * y;
            const double kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2);
            const double u = fx * (x * kr + p1 * 2 * x * y + p2 * (r2 + 2 * x * x)) + cx;
            const double v = fy * (y * kr + p1 * (r2 + 2 * y * y) + p2 * 2 * x * y) + cy;
            const int iu = lens_round(u * 32), iv = lens_round(v * 32);
            const size_t o = (size_t)i * cols + j;
            xy[2 * o] = lens_sat16(iu >> 5);
            xy[2 * o + 1] = lens_sat16(iv >> 5);
            fr[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
        }
}

void orc_fisheye_map(int rows, int cols, const double K[9], const double D[4], const double Knew[9], int16_t* xy, uint16_t* fr)
{
    const double fx = K[0], fy = K[4], cx = K[2], cy = K[5];
    const double nfx = Knew[0], nfy = Knew[4], ncx = Knew[2], ncy = Knew[5];
    for (int i = 0; i < rows; ++i)
        for (int j = 0; j < cols; ++j) {
            const double x = (j - ncx) / nfx, y = (i - ncy) / nfy;
            const double r = sqrt(x * x + y * y);
            const double th = atan(r);
            const double th2 = th * th, th4 = th2 * th2, th6 = th4 * th2, th8 = th4 * th4;
            const double thd = th * (1 + D[0] * th2 + D[1] * th4 + D[2] * th6 + D[3] * th8);
            const double s = r == 0 ? 1.0 : thd / r;
            const double u = fx * x * s + cx, v = fy * y * s + cy;
            const int iu = lens_round(u * 32), iv = lens_round(v * 32);
            const size_t o = (size_t)i * cols + j;
            xy[2 * o] = (int16_t)(uint16_t)(unsigned)(iu >> 5);
            xy[2 * o + 1] = (int16_t)(uint16_t)(unsigned)(iv >> 5);
            fr[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
        }
}
