// The v3 tracker's conversions (klt_v3.cuh), in a header of their own so that tests can run them beside the shared
// forms of klt.cu.  Needs W_BITS (klt.cu: 14).
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>

// The kernel's forms of floor_to_int / __float2int_rd and bilinear_weights (klt.cu): FADDs on the FMA pipe instead of
// F2I / I2F on the slow conversion pipe, with the same bits on every input the kernel feeds them.
//
// Floor.  t = RD(x + 1.5 * 2^23).  For x in [-2^22, 2^22) the exact sum lies in [2^23, 2^24), where the floats are the integers,
// so t = 1.5 * 2^23 + floor(x) exactly: its bit pattern is V3_FLOOR_BITS + floor(x), and t - 1.5 * 2^23 is floor(x) as a
// float, exactly (the same float as (float)floor(x), so x minus it is the shared form's fraction bit for bit).  Outside
// that range, non-finite x included, bits - V3_FLOOR_BITS is >= 2^22 or < -2^22: RD is monotone, t >= 2^24 for x >= 2^22 and t < 2^23
// for x < -2^22; a negative t has the sign bit set, which wraps the difference (mod 2^32) to >= 0x34C00000 for t in
// (-1.5 * 2^23, -0] and below -2^30 for t <= -1.5 * 2^23; NaN gives 0x34BFFFFF.  The launch takes this kernel only for
// levels smaller than 2^22 in both dimensions, so exactly those positions fail the range test (or the staged-window
// test) that floor_to_int's INT_MIN, F2I's saturation or the exact floor made fail before.
#define V3_FLOOR_MAGIC 12582912.f      // 1.5 * 2^23
#define V3_FLOOR_BITS 0x4B400000u      // its bit pattern
__device__ __forceinline__ float floor_v3(float x, uint32_t& bits)
{
    const float t = __fadd_rd(x, V3_FLOOR_MAGIC);
    bits = __float_as_uint(t);
    return __fsub_rn(t, V3_FLOOR_MAGIC);
}
__device__ __forceinline__ int floor_bits_to_int(uint32_t bits) { return (int)(bits - V3_FLOOR_BITS); }

// Weights.  cvRound(p * 2^14) of p in [0, 1] is __float2int_rn of the exactly scaled product.  RN(p + 768) lies in
// [768, 769], inside the binade [512, 1024) whose spacing is 2^-14, so it is 768 + k * 2^-14 with k = p * 2^14 rounded to
// nearest, ties to even (768's significand is even: the parity of the last significand bit is the parity of k).  Its bit
// pattern is 0x44400000 + k with k <= 2^14: the low 16 bits are the weight.  iw11 = 2^14 - iw00 - iw01 - iw10 only
// matters modulo 2^16 (a signed 16-bit half, -1 included: DESIGN §2 fact 6), where 3 * 0x44400000 vanishes, so it comes
// straight from the bit patterns.  wt = iw00 | iw01 << 16 and wb = iw10 | iw11 << 16, as interp_run8_64 takes them.
__device__ __forceinline__ void bilinear_weights_v3(float a, float b, uint32_t& wt, uint32_t& wb)
{
    const float a1 = __fsub_rn(1.f, a), b1 = __fsub_rn(1.f, b);
    const uint32_t p00 = __float_as_uint(__fadd_rn(__fmul_rn(a1, b1), 768.f));
    const uint32_t p01 = __float_as_uint(__fadd_rn(__fmul_rn(a, b1), 768.f));
    const uint32_t p10 = __float_as_uint(__fadd_rn(__fmul_rn(a1, b), 768.f));
    const uint32_t w11 = (1u << W_BITS) - p00 - p01 - p10;
    wt = __byte_perm(p00, p01, 0x5410);
    wb = __byte_perm(p10, w11, 0x5410);
}

// RN(x / d) is monotone in x, so minEig = RN(num / (2 * WW * WH)) < thr holds exactly for the floats num below one
// boundary: the smallest float x (in the order -inf < ... < -0 < +0 < ... < +inf) with !(RN(x / d) < thr).  -0 and +0
// give quotients that compare equal, so num < boundary decides both alike.  Found by bisection over the float order on
// the host (IEEE division there is the same correctly rounded RN(x / d) as __fdiv_rn).
static inline float min_eig_num_bound(float thr, float d)
{
    auto key = [](float f) { int32_t u; memcpy(&u, &f, 4); return u < 0 ? -(int64_t)(u & 0x7FFFFFFF) - 1 : (int64_t)u; };
    auto val = [](int64_t k) { const int32_t u = k < 0 ? (int32_t)((-k - 1) | 0x80000000ll) : (int32_t)k; float f; memcpy(&f, &u, 4); return f; };
    auto pass = [&](int64_t k) { volatile float q = val(k) / d; return !(q < thr); };
    int64_t lo = key(-INFINITY), hi = key(INFINITY);   // pass(hi) always holds: inf < thr never does
    if (pass(lo)) return -INFINITY;
    while (hi - lo > 1) {   // invariant: !pass(lo), pass(hi)
        const int64_t mid = lo + (hi - lo) / 2;
        (pass(mid) ? hi : lo) = mid;
    }
    return val(hi);
}
