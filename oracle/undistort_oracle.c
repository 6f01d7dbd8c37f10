/* cv2.undistort(src, K, dist) with newCameraMatrix = K, restated (test-only CPU oracle):
 *   map:   cv2.initUndistortRectifyMap(K, dist, None, K, (cols, rows), CV_16SC2), evaluated in plain double over the whole
 *          frame (cv2 evaluates it in stripes; rounding to 1/32 px gives the same entries) -- int16 source pixel, saturated,
 *          and the fraction (v & 31) * 32 + (u & 31);
 *   remap: cv2.remap(src, map, INTER_LINEAR, BORDER_CONSTANT 0) in fixed point, each tap outside the image contributing 0.
 * dist: the 8 coefficients k1, k2, p1, p2, k3, k4, k5, k6 (shorter models padded with zeros). */
#include <math.h>
#include <limits.h>
#include <stddef.h>
#include <stdint.h>

/* cvRound on x86 (cvtsd2si): NaN, +-inf and values outside int32 give INT_MIN */
static int und_round(double a)
{
    if (!(a > -2147483648.5 && a < 2147483647.5)) return INT_MIN;
    return (int)rint(a);
}

static int16_t und_sat16(int v) { return (int16_t)(v < -32768 ? -32768 : v > 32767 ? 32767 : v); }

void orc_undistort_map(int rows, int cols, const double K[9], const double d[8], int16_t* xy, uint16_t* fr)
{
    const double fx = K[0], fy = K[4], cx = K[2], cy = K[5];
    const double k1 = d[0], k2 = d[1], p1 = d[2], p2 = d[3], k3 = d[4], k4 = d[5], k5 = d[6], k6 = d[7];
    for (int i = 0; i < rows; ++i)
        for (int j = 0; j < cols; ++j) {
            const double x = (j - cx) / fx, y = (i - cy) / fy;
            const double r2 = x * x + y * y;
            const double kr = (1 + ((k3 * r2 + k2) * r2 + k1) * r2) / (1 + ((k6 * r2 + k5) * r2 + k4) * r2);
            const double u = fx * (x * kr + p1 * 2 * x * y + p2 * (r2 + 2 * x * x)) + cx;
            const double v = fy * (y * kr + p1 * (r2 + 2 * y * y) + p2 * 2 * x * y) + cy;
            const int iu = und_round(u * 32), iv = und_round(v * 32);
            const size_t o = (size_t)i * cols + j;
            xy[2 * o] = und_sat16(iu >> 5);
            xy[2 * o + 1] = und_sat16(iv >> 5);
            fr[o] = (uint16_t)((iv & 31) * 32 + (iu & 31));
        }
}

void orc_remap_linear(const uint8_t* src, int rows, int cols, const int16_t* xy, const uint16_t* fr, uint8_t* dst)
{
    for (int i = 0; i < rows; ++i)
        for (int j = 0; j < cols; ++j) {
            const size_t o = (size_t)i * cols + j;
            const int sx = xy[2 * o], sy = xy[2 * o + 1], ax = fr[o] & 31, ay = fr[o] >> 5;
            int t[4];
            for (int k = 0; k < 4; ++k) {
                const int xx = sx + (k & 1), yy = sy + (k >> 1);
                t[k] = (xx >= 0 && xx < cols && yy >= 0 && yy < rows) ? src[(size_t)yy * cols + xx] : 0;
            }
            const int s = 32 * (t[0] * (32 - ax) * (32 - ay) + t[1] * ax * (32 - ay) + t[2] * (32 - ax) * ay + t[3] * ax * ay);
            dst[o] = (uint8_t)((s + (1 << 14)) >> 15);
        }
}
