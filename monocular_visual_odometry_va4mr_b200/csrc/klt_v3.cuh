// klt_kernel_v3<WW,WH>: the tracker for the two window sizes the workloads use (15x15: the reference's
// options, main.py:36; 21x21: cv2's default).  Same arithmetic as klt_kernel, bit-identical results:
//   * a lane owns a run of 8 horizontally adjacent window pixels (row y, x0 = 0, 8, 16) instead of every
//     32nd pixel, read with two LDS.64 per row from rows of 40 bytes (5 eight-byte slots) and re-aligned
//     with funnel shifts: with lanes 0-15 on the left runs and lanes 16-31 on the right runs each half-warp
//     touches 15 distinct slots, so the window reads are conflict-free;
//   * the bilinear interpolation I00*w00 + I01*w01 (+ next row) is two dp2a (16-bit weights x 8-bit pixels)
//     instead of four IMAD; the template gradients are Scharr of the unrounded bilinear image when the window's tap
//     grid lies inside the image (template_interior), otherwise 5 dp4a per tap on the staged patch, interpolated;
//   * the window of the NEXT image is staged in shared memory per level by 8-byte cp.async (window + 4 px
//     margin, restaged only if the point leaves it), so iterations never touch L1/L2;
//   * the template gradients live in registers; sum(Iwin*dI) is folded into two constants, so an iteration
//     needs neither Iwin nor a subtraction per pixel;
//   * PERSISTENT warps + an atomic work queue (SURVEY 7.3): a warp fetches the next feature when its own
//     converges, so a CTA slot is never held by the slowest of four features, and small shards (8 sequences
//     per GPU in the strong-scaling run) are not tail-bound (profiles/r2a_klt_source_hot.txt);
//   * iteration loop: the staged-window test and the image-range test are ONE unsigned compare per axis
//     against bounds fixed at staging time; floor and cvRound by magic-constant FADDs instead of F2I / I2F, the
//     packed weights straight from their bit patterns (klt_v3_forms.cuh); the two exact 64-bit warp sums take a
//     single-REDUX fast path when a per-level bound rules out an int32 overflow (ITER_SUM_FAST_MAX; the hi/lo
//     split path is kept for the rest);
//   * level setup: the minEig test is a compare of its numerator against a bound found on the host (no division);
//   * Iwin and the final error pass are skipped when the point set has no error output.
#pragma once
#include <type_traits>
#include "klt_v3_forms.cuh"

// 16-bit weights x 8-bit pixels.  The weights are SIGNED halves: iw11 = 2^14 - iw00 - iw01 - iw10 is -1
// when the three rounded weights add up to 2^14 + 1 (a fractional part of ~0 in x or y, about one
// position in a thousand) -- cv2 carries that -1 through its integer arithmetic, and so must this.
__device__ __forceinline__ uint32_t dp2a_lo_u(uint32_t a, uint32_t b, uint32_t c)
{
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"((int)c));
    return (uint32_t)d;
}
__device__ __forceinline__ uint32_t dp2a_hi_u(uint32_t a, uint32_t b, uint32_t c)
{
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"((int)c));
    return (uint32_t)d;
}
__device__ __forceinline__ int dp4a_us(uint32_t a, int b, int c)   // unsigned pixels x signed coefficients
{
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

// asynchronous global -> shared staging (LDGSTS): the copy proceeds while the warp computes
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_pending(int n)   // wait until at most n groups are pending
{
    if (n <= 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
    else if (n == 1) asm volatile("cp.async.wait_group 1;" ::: "memory");
    else asm volatile("cp.async.wait_group 2;" ::: "memory");
}

template <int WW, int WH>
struct KV3 {
    static constexpr int NSEG = (WW + 7) / 8;            // 8-pixel runs per window row
    static constexpr bool SPLIT = NSEG == 2 && WH <= 16; // lanes 0-15: left runs, lanes 16-31: right runs
    static constexpr int NTASK = WH * NSEG;
    static constexpr int NROUND = SPLIT ? 1 : (NTASK + 31) / 32;
    static constexpr int DW = WW + 1, DH = WH + 1;       // derivative tap grid
    static constexpr int DSEG = (DW + 7) / 8;
    static constexpr int DTASK = DH * DSEG;
    static constexpr int DROUND = (DTASK + 31) / 32;
    static constexpr int DS = ((NSEG * 8 + 1 + 3) / 4) * 4 > DSEG * 8 ? ((NSEG * 8 + 1 + 3) / 4) * 4 : DSEG * 8;  // ints per der row
    static constexpr int MARGIN = 4;
    static constexpr int odd_slots(int bytes) { return ((bytes + 7) / 8) % 2 == 0 ? (bytes + 7) / 8 + 1 : (bytes + 7) / 8; }
    static constexpr int PSLOT = odd_slots(7 + WW + 3);              // 8-byte slots per patch row (odd: rows spread over the banks)
    static constexpr int PS = PSLOT * 8;
    static constexpr int PROWS = WH + 3;
    static constexpr int JSLOT = odd_slots(7 + WW + 1 + 2 * MARGIN + 1);
    static constexpr int JS = JSLOT * 8;
    static constexpr int JR = WH + 1 + 2 * MARGIN;
    static constexpr int IS = NSEG * 8;                   // Iwin row stride (shorts)
    static constexpr int B_PATCH = ((PS * PROWS + 16 + 15) / 16) * 16;
    static constexpr int B_J = ((JS * JR + 16 + 15) / 16) * 16;
    static constexpr int B_DER = DS * DH * 4;             // per plane
    static constexpr int B_IWIN = ((IS * WH * 2 + 15) / 16) * 16;
    static constexpr int PER_WARP = 2 * B_PATCH + B_J + 2 * B_DER + B_IWIN;   // two patch buffers (prefetch)
    static constexpr int MIN_CTAS = ((227 * 1024) / (KLT_WARPS * PER_WARP + 64 + 1024) * KLT_WARPS >= 32 ? 32 : 24) / KLT_WARPS;
    // An iteration's lane partial is sum (IvJ - Iwin) * dIx over the lane's 8 * NROUND pixels, with IvJ and Iwin in
    // [0, 8160]; by Cauchy-Schwarz |partial| <= 8160 * sqrt(8 * NROUND * sum dIx^2).  A lane sum of dIx^2 (and of
    // dIy^2) up to this bound keeps every partial of the level below 2^26: the single-REDUX sums are exact.
    static constexpr int ITER_SUM_FAST_MAX = (int)(((1ll << 52) - 1) / (8160ll * 8160ll * (8 * NROUND)));
};

__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void cp_async8(uint32_t smem_dst, const void* gsrc)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
// Rows of SPR eight-byte slots; each lane owns a fixed (row-in-round, slot): 32 / SPR rows per round.
template <int SPR, int ROWS>
__device__ __forceinline__ void stage_rows_async8(uint32_t dst_s, const uint8_t* src_aligned, int pitch, int lane)
{
    constexpr int RPR = 32 / SPR;
    const int r0 = lane / SPR, c = lane - r0 * SPR;
    if (r0 >= RPR) return;
    const uint8_t* src = src_aligned + (long long)r0 * pitch + c * 8;
    uint32_t d = dst_s + (uint32_t)(r0 * SPR + c) * 8u;
    const long long sstep = (long long)RPR * pitch;
#pragma unroll
    for (int r = 0; r < (ROWS + RPR - 1) / RPR; ++r) {
        if (r * RPR + r0 < ROWS) cp_async8(d, src);
        src += sstep;
        d += RPR * SPR * 8;
    }
}

__device__ __forceinline__ uint2 lds_u64(uint32_t addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}

// 8 interpolated intensities (13-bit, = 32 x grey level) of the run starting at byte offset `off` of the row at
// shared address `img_s` (and the row RS bytes below it).  HI = bit 2 of off (warp-uniform, hoisted by the caller);
// sh8 = (off & 3) * 8.  wt = iw00 | iw01 << 16, wb = iw10 | iw11 << 16 (signed 16-bit halves).
template <int RS, bool HI>
__device__ __forceinline__ void interp_run8_64(uint32_t img_s, int off, int sh8, uint32_t wt, uint32_t wb, int* I)
{
    const uint32_t t = img_s + (uint32_t)(off & ~7), b = t + RS;
    const uint2 tA = lds_u64(t), tB = lds_u64(t + 8), bA = lds_u64(b), bB = lds_u64(b + 8);
    const uint32_t t0 = HI ? tA.y : tA.x, t1 = HI ? tB.x : tA.y, t2 = HI ? tB.y : tB.x;
    const uint32_t b0 = HI ? bA.y : bA.x, b1 = HI ? bB.x : bA.y, b2 = HI ? bB.y : bB.x;
    const uint32_t ta0 = __funnelshift_r(t0, t1, sh8), ta1 = __funnelshift_r(t1, t2, sh8), ta2 = t2 >> sh8;
    const uint32_t ba0 = __funnelshift_r(b0, b1, sh8), ba1 = __funnelshift_r(b1, b2, sh8), ba2 = b2 >> sh8;
    const uint32_t ts0 = __funnelshift_r(ta0, ta1, 8), ts1 = __funnelshift_r(ta1, ta2, 8);
    const uint32_t bs0 = __funnelshift_r(ba0, ba1, 8), bs1 = __funnelshift_r(ba1, ba2, 8);
    const uint32_t R = 1u << (W_BITS - 5 - 1);
    I[0] = (int)(dp2a_lo_u(wb, ba0, dp2a_lo_u(wt, ta0, R)) >> (W_BITS - 5));
    I[1] = (int)(dp2a_lo_u(wb, bs0, dp2a_lo_u(wt, ts0, R)) >> (W_BITS - 5));
    I[2] = (int)(dp2a_hi_u(wb, ba0, dp2a_hi_u(wt, ta0, R)) >> (W_BITS - 5));
    I[3] = (int)(dp2a_hi_u(wb, bs0, dp2a_hi_u(wt, ts0, R)) >> (W_BITS - 5));
    I[4] = (int)(dp2a_lo_u(wb, ba1, dp2a_lo_u(wt, ta1, R)) >> (W_BITS - 5));
    I[5] = (int)(dp2a_lo_u(wb, bs1, dp2a_lo_u(wt, ts1, R)) >> (W_BITS - 5));
    I[6] = (int)(dp2a_hi_u(wb, ba1, dp2a_hi_u(wt, ta1, R)) >> (W_BITS - 5));
    I[7] = (int)(dp2a_hi_u(wb, bs1, dp2a_hi_u(wt, ts1, R)) >> (W_BITS - 5));
}

// Exact sums of two int32 values over the warp, as float32 (== __ll2float_rn of the 64-bit sums).  A lane partial
// below 2^26 in magnitude cannot overflow the 32-lane int32 sum: one REDUX each; otherwise (wide) the hi/lo split
// path.  Both give the same float whenever the single REDUX is exact.
__device__ __forceinline__ void warp_sum2_f32(int v1, int v2, bool wide, float& f1, float& f2)
{
    if (wide) {
        f1 = __ll2float_rn(warp_sum_i64(v1));
        f2 = __ll2float_rn(warp_sum_i64(v2));
    } else {
        f1 = __int2float_rn(__reduce_add_sync(0xffffffffu, v1));
        f2 = __int2float_rn(__reduce_add_sync(0xffffffffu, v2));
    }
}
__device__ __forceinline__ void warp_sum2_f32(int v1, int v2, float& f1, float& f2)
{
    warp_sum2_f32(v1, v2, __any_sync(0xffffffffu, max(abs(v1), abs(v2)) >= (1 << 26)), f1, f2);
}

// Template derivatives of a window whose whole tap grid lies inside the image, for the split layout (lane = window
// row ty = lane & 15, columns tx .. tx+7).  Scharr is linear, so the bilinear blend of Scharr taps equals Scharr of
// the unrounded bilinear image U(u, v) = iw00 p(u,v) + iw01 p(u+1,v) + iw10 p(u,v+1) + iw11 p(u+1,v+1), exactly in
// int32 (|Scharr(U)| <= 16 * 255 * (2^14 + 2) < 2^31).  With no tap zeroed at the image border this is the value
// the tap grid gives, bit for bit.  The lane computes U on rows ty-1 and ty for columns tx-1 .. tx+8 and takes row
// ty+1 from the next lane (the last lane of each half computes row WH for it).  The dp2a chains carry the +2^8 of
// the rounding of Iv; the Scharr kernels sum to zero, so it cancels in the derivatives.
template <bool HI>
__device__ __forceinline__ void patch_row_pairs10(uint32_t addr8, int sh8, uint32_t* w)
{
    const uint2 A = lds_u64(addr8), B = lds_u64(addr8 + 8);
    uint32_t t0, t1, t2, t3;
    if (HI) { const uint2 Cc = lds_u64(addr8 + 16); t0 = A.y; t1 = B.x; t2 = B.y; t3 = Cc.x; }
    else { t0 = A.x; t1 = A.y; t2 = B.x; t3 = B.y; }
    const uint32_t a0 = __funnelshift_r(t0, t1, sh8), a1 = __funnelshift_r(t1, t2, sh8), a2 = __funnelshift_r(t2, t3, sh8);
    w[0] = a0; w[1] = __funnelshift_r(a0, a1, 8); w[2] = a1; w[3] = __funnelshift_r(a1, a2, 8); w[4] = a2; w[5] = a2 >> 8;
}
// U (+2^8) of columns c = 0..9 from the pair words of the row (top) and the row below (bot)
__device__ __forceinline__ void interp_row10(const uint32_t* top, const uint32_t* bot, uint32_t wt, uint32_t wb, int* U)
{
    const uint32_t R = 1u << (W_BITS - 5 - 1);
#pragma unroll
    for (int q = 0; q < 3; ++q) {
        const int c = 4 * q;
        U[c] = (int)dp2a_lo_u(wb, bot[2 * q], dp2a_lo_u(wt, top[2 * q], R));
        U[c + 1] = (int)dp2a_lo_u(wb, bot[2 * q + 1], dp2a_lo_u(wt, top[2 * q + 1], R));
        if (q < 2) {
            U[c + 2] = (int)dp2a_hi_u(wb, bot[2 * q], dp2a_hi_u(wt, top[2 * q], R));
            U[c + 3] = (int)dp2a_hi_u(wb, bot[2 * q + 1], dp2a_hi_u(wt, top[2 * q + 1], R));
        }
    }
}
template <int PS, bool HI>
__device__ __forceinline__ void template_interior(uint32_t patch_s, int row_off, int sh8, uint32_t wt, uint32_t wb,
                                                  int* gx, int* gy, int* Iv)
{
    // row_off: byte of pixel (tx-1, ty-1), rounded down to 8
    uint32_t pa[6], pb[6], pc[6];
    patch_row_pairs10<HI>(patch_s + row_off, sh8, pa);
    patch_row_pairs10<HI>(patch_s + row_off + PS, sh8, pb);
    patch_row_pairs10<HI>(patch_s + row_off + 2 * PS, sh8, pc);
    int Um[10], U0[10];
    interp_row10(pa, pb, wt, wb, Um);
    interp_row10(pb, pc, wt, wb, U0);
    int S[10], D[10];
#pragma unroll
    for (int c = 0; c < 10; ++c) {
        const int Up = __shfl_down_sync(0xffffffffu, U0[c], 1, 16);
        D[c] = Up - Um[c];
        S[c] = (Up + Um[c]) * 3 + U0[c] * 10;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        gx[k] = (S[k + 2] - S[k] + (1 << (W_BITS - 1))) >> W_BITS;
        gy[k] = ((D[k] + D[k + 2]) * 3 + D[k + 1] * 10 + (1 << (W_BITS - 1))) >> W_BITS;
        Iv[k] = (int)((uint32_t)U0[k + 1] >> (W_BITS - 5));
    }
}

// EXT: the sequences have their own level counts and level sizes (a.ext); otherwise a.levels / a.w / a.h hold for all
template <int WW, int WH, bool EXT>
__global__ void __launch_bounds__(KLT_WARPS * 32, (KV3<WW, WH>::MIN_CTAS))
klt_kernel_v3(const KltArgs a)
{
    using C = KV3<WW, WH>;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const int cap_all = a.cap[0] + a.cap[1];
    const int total = a.batch * cap_all;

    uint8_t* wbase = smem + (size_t)warp * C::PER_WARP;
    uint32_t wbase_s;     // opaque to the compiler: stays in a register instead of being rebuilt per use
    asm volatile("mov.u32 %0, %1;" : "=r"(wbase_s) : "r"((uint32_t)__cvta_generic_to_shared(wbase)));
    const uint32_t jreg_s = wbase_s + 2 * C::B_PATCH;
    int* derx = reinterpret_cast<int*>(wbase + 2 * C::B_PATCH + C::B_J);
    int* dery = derx + C::DS * C::DH;
    short* Iwin = reinterpret_cast<short*>(wbase + 2 * C::B_PATCH + C::B_J + 2 * C::B_DER);

    const float hwx = (WW - 1) * 0.5f, hwy = (WH - 1) * 0.5f;
    const float FLT_SCALE = 1.f / (1 << 20);

    // this lane's template runs: (row ty[r], first column tx[r], live pixels tl[r]) per round
    int ty[C::NROUND], tx[C::NROUND], tl[C::NROUND];
#pragma unroll
    for (int r = 0; r < C::NROUND; ++r) {
        if (C::SPLIT) {
            ty[r] = lane & 15;
            tx[r] = (lane >> 4) * 8;
            tl[r] = ty[r] < WH ? min(8, WW - tx[r]) : 0;
            if (ty[r] >= WH) ty[r] = 0;
        } else {
            const int t = r * 32 + lane;
            ty[r] = t / C::NSEG;
            tx[r] = (t - ty[r] * C::NSEG) * 8;
            tl[r] = t < C::NTASK ? min(8, WW - tx[r]) : 0;
            if (t >= C::NTASK) { ty[r] = 0; tx[r] = 0; }
        }
    }
    // split layout: the live pixels of the lane's run as masks, the first WW - 8 (live in both runs of a live row) and
    // the rest (live in a left run of a live row only)
    const int mrow = tl[0] > 0 ? -1 : 0, mtail = tl[0] == 8 ? -1 : 0;
    // this lane's byte offsets inside the staged J window, pinned to registers
    int joffl[C::NROUND];
#pragma unroll
    for (int r = 0; r < C::NROUND; ++r) asm volatile("mov.s32 %0, %1;" : "=r"(joffl[r]) : "r"(ty[r] * C::JS + tx[r]));
    const float eps_lo = a.eps_lo, eps_hi = a.eps_hi;

    // ---- work queue: a.queue[0] = next feature slot, a.queue[1] = warps that found the queue empty ----
    // The next slot is fetched one feature ahead (the atomic's round trip hides behind the feature) only when the launch
    // has at least two features per warp: in a small launch (a single sequence: 1000 features for 1000 warps) fetching
    // ahead lets the first half of the warps claim two features each while the other half of the machine gets none.
    const bool ahead = total >= 2 * (int)gridDim.x * KLT_WARPS;
    int gw = 0;
    if (lane == 0) {
        gw = atomicAdd(a.queue, 1);
        if (gw == 0) reinterpret_cast<unsigned long long*>(a.queue)[1] = global_timer_ns();   // trace: first feature claimed
    }
    gw = __shfl_sync(0xffffffffu, gw, 0);
    while (gw < total) {
        int gw_next = 0;
        if (ahead && lane == 0) gw_next = atomicAdd(a.queue, 1);   // fetched now, consumed when this feature is done
        const int seq = gw / cap_all;
        int pi = gw - seq * cap_all;
        const int seg = pi >= a.cap[0] ? 1 : 0;
        pi -= seg ? a.cap[0] : 0;
        const int n_here = a.n_pts[seg] ? min(a.n_pts[seg][seq], a.cap[seg]) : a.n_fixed;
        if (pi < n_here) {
    const uint8_t* prev = a.prev + (size_t)seq * a.prev_stride;
    const uint8_t* next = a.next + (size_t)seq * a.next_stride;
    const size_t pidx = (size_t)seq * a.cap[seg] + pi;
    const float px0 = a.pts[seg][2 * pidx], py0 = a.pts[seg][2 * pidx + 1];
    const bool want_err = a.err[seg] != nullptr;   // Iwin and the final error are only needed for this
    float outx = 0.f, outy = 0.f;
    int st = 1;
    float e = 0.f;
    int pb = 0, pf_level = -1;     // patch buffer in use; level whose patch was prefetched into it
    cp_async_wait_pending(0);      // nothing of the previous feature may still be landing in this warp's buffers
    __syncwarp();
    const VoSeqExt* ext = EXT ? a.ext + seq : nullptr;
    const int levels = EXT ? ext->levels : a.levels;

    for (int level = levels - 1; level >= 0; --level) {
        int lw, lh;
        asm volatile("mov.s32 %0, %1;" : "=r"(lw) : "r"(EXT ? ext->w[level] : a.w[level]));
        asm volatile("mov.s32 %0, %1;" : "=r"(lh) : "r"(EXT ? ext->h[level] : a.h[level]));
        const int pitch = a.pitch[level];
        const uint8_t* I = prev + a.off[level];
        const uint8_t* J = next + a.off[level];
        const float sc = __int_as_float((127 - level) << 23);   // exactly 2^-level
        float ppx = __fmul_rn(px0, sc), ppy = __fmul_rn(py0, sc);
        float nx, ny;
        if (level == levels - 1) { nx = ppx; ny = ppy; }
        else { nx = __fmul_rn(outx, 2.f); ny = __fmul_rn(outy, 2.f); }
        outx = nx; outy = ny;
        ppx = __fsub_rn(ppx, hwx); ppy = __fsub_rn(ppy, hwy);
        uint32_t bpx, bpy;
        const float fpx = floor_v3(ppx, bpx), fpy = floor_v3(ppy, bpy);
        const int ipx = floor_bits_to_int(bpx), ipy = floor_bits_to_int(bpy);
        if (ipx < -WW || ipx >= lw || ipy < -WH || ipy >= lh) {
            if (level == 0) { st = 0; e = 0.f; }
            continue;
        }
        // wt = iw00 | iw01 << 16, wb = iw10 | iw11 << 16.  The layouts of more than two runs per row (21x21) take every
        // template through the per-tap path, which wants the four weights as integers: there the packed form costs a
        // spill at 80 registers, so they keep the shared helper (the same weights)
        uint32_t wt, wb;
        int iw00, iw01, iw10, iw11;
        if (C::SPLIT) {
            bilinear_weights_v3(__fsub_rn(ppx, fpx), __fsub_rn(ppy, fpy), wt, wb);
            iw00 = (int)(wt & 0xFFFF); iw01 = (int)(wt >> 16); iw10 = (int)(wb & 0xFFFF); iw11 = (int)wb >> 16;
        } else {
            bilinear_weights(__fsub_rn(ppx, fpx), __fsub_rn(ppy, fpy), iw00, iw01, iw10, iw11);
            wt = (uint32_t)(iw01 * 65536 + iw00); wb = (uint32_t)iw11 * 65536u + (uint32_t)iw10;
        }

        // ---- staging pipeline (cp.async): this level's patch of I was prefetched during the previous
        // level; now start (1) the window of J around the initial position and (2) the NEXT level's
        // patch of I (its position depends only on the input point), and overlap both with the
        // derivative / template arithmetic of this level ----
        __syncwarp();
        const uint32_t patch_s = wbase_s + pb * C::B_PATCH;
        const uint8_t* patch = wbase + pb * C::B_PATCH;
        const uint8_t* src0 = I + (long long)(ipy - 1) * pitch + (ipx - 1);
        const int mis = (int)(reinterpret_cast<uintptr_t>(src0) & 7);
        if (pf_level != level) {   // not prefetched (top level, or the previous level was skipped)
            stage_rows_async8<C::PSLOT, C::PROWS>(patch_s, src0 - mis, pitch, lane);
            cp_async_commit();
        }
        const float jx0 = __fsub_rn(nx, hwx), jy0 = __fsub_rn(ny, hwy);
        // staged J window: valid (inx, iny) are xlo + [0, xspan] x ylo + [0, yspan] = inside the window AND inside the
        // image range cv2 accepts, tested on floor_v3's bit patterns: xlob = V3_FLOOR_BITS + xlo (mod 2^32); jbase = byte
        // offset of (xlo, ylo) in the window.  Nothing staged: the test always fails -- the sentinel is the pattern of
        // -3.7e-32, and RD(x + 1.5 * 2^23) is +-0 or at least 0.5 in magnitude (x and 1.5 * 2^23 are multiples of 0.5
        // wherever they can cancel)
        uint32_t xlob = 0x8B400001u, ylob = 0x8B400001u;
        int jbase = 0;
        unsigned xspan = 0, yspan = 0;
        auto stage_J = [&](int inx, int iny) {
            const int ry0 = iny - C::MARGIN;
            const uint8_t* s0 = J + (long long)ry0 * pitch + (inx - C::MARGIN);
            const int m2 = (int)(reinterpret_cast<uintptr_t>(s0) & 7);
            const int rx0 = inx - C::MARGIN - m2;
            stage_rows_async8<C::JSLOT, C::JR>(jreg_s, s0 - m2, pitch, lane);
            const int xlo = max(rx0, -WW), ylo = max(ry0, -WH);
            const int xhi = min(rx0 + C::JS - WW - 2, lw - 1), yhi = min(ry0 + C::JR - WH - 2, lh - 1);
            xspan = (unsigned)(xhi - xlo); yspan = (unsigned)(yhi - ylo);     // the staging position itself is valid: spans >= 0
            xlob = (uint32_t)xlo + V3_FLOOR_BITS; ylob = (uint32_t)ylo + V3_FLOOR_BITS;
            jbase = (ylo - ry0) * C::JS + (xlo - rx0);
        };
        {
            uint32_t bx, by;
            floor_v3(jx0, bx); floor_v3(jy0, by);
            const int inx = floor_bits_to_int(bx), iny = floor_bits_to_int(by);
            if (!(inx < -WW || inx >= lw || iny < -WH || iny >= lh)) stage_J(inx, iny);
            cp_async_commit();
        }
        bool pf_next = false;
        if (level > 0) {
            const int nl = level - 1;
            const float sc2 = __int_as_float((127 - nl) << 23);
            uint32_t bx, by;
            floor_v3(__fsub_rn(__fmul_rn(px0, sc2), hwx), bx); floor_v3(__fsub_rn(__fmul_rn(py0, sc2), hwy), by);
            const int qx = floor_bits_to_int(bx), qy = floor_bits_to_int(by);
            if (!(qx < -WW || qx >= (EXT ? ext->w[nl] : a.w[nl]) || qy < -WH || qy >= (EXT ? ext->h[nl] : a.h[nl]))) {
                const uint8_t* n0 = prev + a.off[nl] + (long long)(qy - 1) * a.pitch[nl] + (qx - 1);
                const int m3 = (int)(reinterpret_cast<uintptr_t>(n0) & 7);
                stage_rows_async8<C::PSLOT, C::PROWS>(wbase_s + (pb ^ 1) * C::B_PATCH, n0 - m3, a.pitch[nl], lane);
                pf_next = true;
            }
            cp_async_commit();
        }
        cp_async_wait_pending(level > 0 ? 2 : 1);   // everything older than (J, next patch): this level's patch
        __syncwarp();
        // patch pixel (x, y), x in [-1, WW+1], y in [-1, WH+1], lives at byte (y+1)*PS + mis + 1 + x

        // ---- template: dIx/dIy (registers), normal matrix, sum(Iwin*dI), Iwin (smem, only for the error) ----
        int gxr[C::NROUND][8], gyr[C::NROUND][8];
        int sA11 = 0, sA12 = 0, sA22 = 0, c1 = 0, c2 = 0;
        auto accumulate = [&](int r, const int* ix, const int* iy, const int* Iv) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                int ixv, iyv;
                if (C::SPLIT) {
                    const int m = k < WW - 8 ? mrow : mtail;
                    ixv = ix[k] & m; iyv = iy[k] & m;
                } else {
                    const bool livek = k < tl[r];
                    ixv = livek ? ix[k] : 0; iyv = livek ? iy[k] : 0;
                }
                gxr[r][k] = ixv; gyr[r][k] = iyv;
                sA11 += ixv * ixv; sA12 += ixv * iyv; sA22 += iyv * iyv;
                c1 += Iv[k] * ixv; c2 += Iv[k] * iyv;
            }
            if (want_err && tl[r] > 0) {
                uint4 pk;
                pk.x = (uint16_t)Iv[0] | ((uint32_t)(uint16_t)Iv[1] << 16); pk.y = (uint16_t)Iv[2] | ((uint32_t)(uint16_t)Iv[3] << 16);
                pk.z = (uint16_t)Iv[4] | ((uint32_t)(uint16_t)Iv[5] << 16); pk.w = (uint16_t)Iv[6] | ((uint32_t)(uint16_t)Iv[7] << 16);
                *reinterpret_cast<uint4*>(Iwin + ty[r] * C::IS + tx[r]) = pk;
            }
        };
        // the whole tap grid (pixels ip + [0, WW] x [0, WH]) inside the image: no tap is zeroed
        if (C::SPLIT && ipx >= 0 && ipx + WW < lw && ipy >= 0 && ipy + WH < lh) {
            const int off = (lane & 15) * C::PS + mis + tx[0];   // byte of pixel (tx-1, row-1); off & 7 == mis
            int ix[8], iy[8], Iv[8];
            if (off & 4) template_interior<C::PS, true>(patch_s, off & ~7, (off & 3) * 8, wt, wb, ix, iy, Iv);
            else template_interior<C::PS, false>(patch_s, off & ~7, (off & 3) * 8, wt, wb, ix, iy, Iv);
            accumulate(0, ix, iy, Iv);
        } else {
            // ---- Scharr on the tap grid: 5 dp4a per pixel, zero outside the image ----
#pragma unroll
            for (int r = 0; r < C::DROUND; ++r) {
                const int t = r * 32 + lane;
                if (t < C::DTASK) {
                    const int gy = t / C::DSEG, gx0 = (t - gy * C::DSEG) * 8;
                    const int off = gy * C::PS + mis + gx0;      // byte of pixel (gx0-1, gy-1)
                    const int sh8 = (off & 3) * 8;
                    int ix[8], iy[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) { ix[k] = 0; iy[k] = 0; }
#pragma unroll
                    for (int rr = 0; rr < 3; ++rr) {
                        const uint32_t* w = reinterpret_cast<const uint32_t*>(patch + (off & ~3) + rr * C::PS);
                        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
                        const uint32_t a0 = __funnelshift_r(w0, w1, sh8), a1 = __funnelshift_r(w1, w2, sh8), a2 = __funnelshift_r(w2, w3, sh8);
                        uint32_t q[8];
                        q[0] = a0; q[1] = __funnelshift_r(a0, a1, 8); q[2] = __funnelshift_r(a0, a1, 16); q[3] = __funnelshift_r(a0, a1, 24);
                        q[4] = a1; q[5] = __funnelshift_r(a1, a2, 8); q[6] = __funnelshift_r(a1, a2, 16); q[7] = __funnelshift_r(a1, a2, 24);
                        // q[k] = pixels (x-1, x, x+1, x+2) of row gy-1+rr for x = gx0+k
                        const int cx = rr == 1 ? 0x000A00F6 : 0x000300FD;                  // (-10,0,10,0) / (-3,0,3,0)
                        const int cy = rr == 0 ? 0x00FDF6FD : 0x00030A03;                  // (-3,-10,-3,0) / (3,10,3,0)
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            ix[k] = dp4a_us(q[k], cx, ix[k]);
                            if (rr != 1) iy[k] = dp4a_us(q[k], cy, iy[k]);
                        }
                    }
                    const int X0 = ipx + gx0, Y = ipy + gy;
                    const bool rowok = Y >= 0 && Y < lh;
                    if (!(rowok && X0 >= 0 && X0 + 7 < lw)) {
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            const bool ok = rowok && X0 + k >= 0 && X0 + k < lw;
                            ix[k] = ok ? ix[k] : 0; iy[k] = ok ? iy[k] : 0;
                        }
                    }
                    int4* dxp = reinterpret_cast<int4*>(derx + gy * C::DS + gx0);
                    int4* dyp = reinterpret_cast<int4*>(dery + gy * C::DS + gx0);
                    dxp[0] = make_int4(ix[0], ix[1], ix[2], ix[3]); dxp[1] = make_int4(ix[4], ix[5], ix[6], ix[7]);
                    dyp[0] = make_int4(iy[0], iy[1], iy[2], iy[3]); dyp[1] = make_int4(iy[4], iy[5], iy[6], iy[7]);
                }
            }
            __syncwarp();
#pragma unroll
            for (int r = 0; r < C::NROUND; ++r) {
                const int off = (ty[r] + 1) * C::PS + mis + 1 + tx[r];
                int Iv[8];
                if (off & 4) interp_run8_64<C::PS, true>(patch_s, off, (off & 3) * 8, wt, wb, Iv);
                else interp_run8_64<C::PS, false>(patch_s, off, (off & 3) * 8, wt, wb, Iv);
                const int* d0 = derx + ty[r] * C::DS + tx[r];
                const int* e0 = dery + ty[r] * C::DS + tx[r];
                int dx0[9], dx1[9], dy0[9], dy1[9];
                {
                    const int4 p0 = *reinterpret_cast<const int4*>(d0), p1 = *reinterpret_cast<const int4*>(d0 + 4);
                    const int4 q0 = *reinterpret_cast<const int4*>(d0 + C::DS), q1 = *reinterpret_cast<const int4*>(d0 + C::DS + 4);
                    dx0[0] = p0.x; dx0[1] = p0.y; dx0[2] = p0.z; dx0[3] = p0.w; dx0[4] = p1.x; dx0[5] = p1.y; dx0[6] = p1.z; dx0[7] = p1.w; dx0[8] = d0[8];
                    dx1[0] = q0.x; dx1[1] = q0.y; dx1[2] = q0.z; dx1[3] = q0.w; dx1[4] = q1.x; dx1[5] = q1.y; dx1[6] = q1.z; dx1[7] = q1.w; dx1[8] = d0[C::DS + 8];
                    const int4 r0 = *reinterpret_cast<const int4*>(e0), r1 = *reinterpret_cast<const int4*>(e0 + 4);
                    const int4 s0 = *reinterpret_cast<const int4*>(e0 + C::DS), s1 = *reinterpret_cast<const int4*>(e0 + C::DS + 4);
                    dy0[0] = r0.x; dy0[1] = r0.y; dy0[2] = r0.z; dy0[3] = r0.w; dy0[4] = r1.x; dy0[5] = r1.y; dy0[6] = r1.z; dy0[7] = r1.w; dy0[8] = e0[8];
                    dy1[0] = s0.x; dy1[1] = s0.y; dy1[2] = s0.z; dy1[3] = s0.w; dy1[4] = s1.x; dy1[5] = s1.y; dy1[6] = s1.z; dy1[7] = s1.w; dy1[8] = e0[C::DS + 8];
                }
                int ix[8], iy[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    ix[k] = (dx0[k] * iw00 + dx0[k + 1] * iw01 + dx1[k] * iw10 + dx1[k + 1] * iw11 + (1 << (W_BITS - 1))) >> W_BITS;
                    iy[k] = (dy0[k] * iw00 + dy0[k + 1] * iw01 + dy1[k] * iw10 + dy1[k + 1] * iw11 + (1 << (W_BITS - 1))) >> W_BITS;
                }
                accumulate(r, ix, iy, Iv);
            }
        }
        const bool wide = __any_sync(0xffffffffu, max(sA11, sA22) > C::ITER_SUM_FAST_MAX);   // this level's iteration sums
        float A11, A12, A22, unused;
        warp_sum2_f32(sA11, sA22, A11, A22);
        warp_sum2_f32(sA12, 0, A12, unused);
        A11 = __fmul_rn(A11, FLT_SCALE); A12 = __fmul_rn(A12, FLT_SCALE); A22 = __fmul_rn(A22, FLT_SCALE);
        float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        const float dA = __fsub_rn(A11, A22);
        // minEig = num / (2 * WW * WH); minEig < min_eig_thr is num < min_eig_num (min_eig_num_bound)
        const float num = __fsub_rn(__fadd_rn(A22, A11),
                                    __fsqrt_rn(__fadd_rn(__fmul_rn(dA, dA), __fmul_rn(__fmul_rn(4.f, A12), A12))));
        // the prefetched patch becomes the current one at the next level, whatever happens below
        if (pf_next) { pb ^= 1; pf_level = level - 1; }
        if (num < a.min_eig_num || D < 1.192092896e-07f) {
            if (level == 0) st = 0;
            cp_async_wait_pending(level > 0 ? 1 : 0);   // drain the J window copy before jreg is reused
            continue;
        }
        D = __fdiv_rn(1.f, D);
        nx = jx0; ny = jy0;
        float pdx = 0.f, pdy = 0.f;
        cp_async_wait_pending(level > 0 ? 1 : 0);   // the window of J has landed (the next patch may still fly)
        __syncwarp();

        for (int j = 0; j < a.max_count; ++j) {
            // cvFloor's INT_MIN, F2I's saturation and floor_v3 all land out of range where one of them does (floor_v3)
            uint32_t bx, by;
            const float fx = floor_v3(nx, bx), fy = floor_v3(ny, by);
            unsigned ux = bx - xlob, uy = by - ylob;
            if (ux > xspan || uy > yspan) {
                const int inx = floor_bits_to_int(bx), iny = floor_bits_to_int(by);
                if (inx < -WW || inx >= lw || iny < -WH || iny >= lh) {
                    if (level == 0) st = 0;
                    break;
                }
                // (re)stage the window of J with a margin around the current position
                __syncwarp();
                stage_J(inx, iny);
                cp_async_commit();
                cp_async_wait_pending(0);
                __syncwarp();
                ux = bx - xlob; uy = by - ylob;
            }
            uint32_t jt, jb;
            bilinear_weights_v3(__fsub_rn(nx, fx), __fsub_rn(ny, fy), jt, jb);
            const int joff = (int)uy * C::JS + (int)ux + jbase;
            int sb1 = -c1, sb2 = -c2;
            const int sh8 = (joff & 3) * 8;
            if (joff & 4) {
#pragma unroll
                for (int r = 0; r < C::NROUND; ++r) {
                    int Iv[8];
                    interp_run8_64<C::JS, true>(jreg_s, joff + joffl[r], sh8, jt, jb, Iv);
#pragma unroll
                    for (int k = 0; k < 8; ++k) { sb1 += Iv[k] * gxr[r][k]; sb2 += Iv[k] * gyr[r][k]; }
                }
            } else {
#pragma unroll
                for (int r = 0; r < C::NROUND; ++r) {
                    int Iv[8];
                    interp_run8_64<C::JS, false>(jreg_s, joff + joffl[r], sh8, jt, jb, Iv);
#pragma unroll
                    for (int k = 0; k < 8; ++k) { sb1 += Iv[k] * gxr[r][k]; sb2 += Iv[k] * gyr[r][k]; }
                }
            }
            float b1, b2;
            warp_sum2_f32(sb1, sb2, wide, b1, b2);
            b1 = __fmul_rn(b1, FLT_SCALE); b2 = __fmul_rn(b2, FLT_SCALE);
            const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D);
            const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D);
            nx = __fadd_rn(nx, dx); ny = __fadd_rn(ny, dy);
            outx = __fadd_rn(nx, hwx); outy = __fadd_rn(ny, hwy);
            // cv2: delta.ddot(delta) <= eps in double; decided in float unless within 1e-6 of the threshold
            const float s2 = __fmaf_rn(dx, dx, __fmul_rn(dy, dy));
            bool conv = s2 < eps_lo;
            if (!conv && !(s2 > eps_hi))
                conv = __dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)) <= a.eps_sq;
            if (conv) break;
            if (j > 0 && fabsf(__fadd_rn(dx, pdx)) < 0.01f && fabsf(__fadd_rn(dy, pdy)) < 0.01f) {
                outx = __fsub_rn(outx, __fmul_rn(dx, 0.5f));
                outy = __fsub_rn(outy, __fmul_rn(dy, 0.5f));
                break;
            }
            pdx = dx; pdy = dy;
        }

        if (st && level == 0) {
            const float qx = __fsub_rn(outx, hwx), qy = __fsub_rn(outy, hwy);
            uint32_t bx, by;
            const float fx = floor_v3(qx, bx), fy = floor_v3(qy, by);
            const int inx = floor_bits_to_int(bx), iny = floor_bits_to_int(by);
            if (inx < -WW || inx >= lw || iny < -WH || iny >= lh) {
                st = 0;
                continue;
            }
            if (!want_err) continue;
            uint32_t jt, jb;
            bilinear_weights_v3(__fsub_rn(qx, fx), __fsub_rn(qy, fy), jt, jb);
            unsigned ux = bx - xlob, uy = by - ylob;
            if (ux > xspan || uy > yspan) {
                __syncwarp();
                stage_J(inx, iny);
                cp_async_commit();
                cp_async_wait_pending(0);
                __syncwarp();
                ux = bx - xlob; uy = by - ylob;
            }
            const int joff = (int)uy * C::JS + (int)ux + jbase;
            int se = 0;
#pragma unroll
            for (int r = 0; r < C::NROUND; ++r) {
                const int off = joff + joffl[r];
                int Iv[8];
                if (off & 4) interp_run8_64<C::JS, true>(jreg_s, off, (off & 3) * 8, jt, jb, Iv);
                else interp_run8_64<C::JS, false>(jreg_s, off, (off & 3) * 8, jt, jb, Iv);
                const uint4 pk = *reinterpret_cast<const uint4*>(Iwin + ty[r] * C::IS + tx[r]);
                const uint32_t pw4[4] = {pk.x, pk.y, pk.z, pk.w};
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int iwv = (int)(short)((pw4[k >> 1] >> ((k & 1) * 16)) & 0xFFFF);
                    se += (k < tl[r]) ? abs(Iv[k] - iwv) : 0;
                }
            }
            e = __fdiv_rn(__ll2float_rn(warp_sum_i64(se)), (float)(32 * WW * WH));
        }
    }
    if (lane == 0) {
        a.out[seg][2 * pidx] = outx;
        a.out[seg][2 * pidx + 1] = outy;
        a.status[seg][pidx] = (uint8_t)st;
        if (a.err[seg]) a.err[seg][pidx] = e;
    }
        }   // pi < n_here
        if (!ahead && lane == 0) gw_next = atomicAdd(a.queue, 1);
        gw = __shfl_sync(0xffffffffu, gw_next, 0);
    }
    // the last warp of the grid to find the queue empty re-arms it for the next launch that uses this slot
    if (lane == 0) {
        const int nwarps = (int)gridDim.x * KLT_WARPS;
        if (atomicAdd(a.queue + 1, 1) == nwarps - 1) {
            reinterpret_cast<unsigned long long*>(a.queue)[2] = global_timer_ns();                   // trace: last warp retired
            a.queue[0] = 0; a.queue[1] = 0; __threadfence();
        }
    }
}
