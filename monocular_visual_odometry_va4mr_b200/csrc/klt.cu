// Pyramidal Lucas-Kanade tracker: one warp per feature, every pyramid level inside one
// kernel (replaces OpenCV's calcSharrDeriv + LKTrackerInvoker behind
// cv2.calcOpticalFlowPyrLK, reference VisualOdometryPipeLine.py:281,287; spec SURVEY.md
// A.2/A.3).
//
// Per level a warp stages the (win+3)^2 neighbourhood of the previous image in shared
// memory, evaluates the Scharr derivative on the fly (never written to HBM), builds the
// 14-bit fixed-point interpolated template (Iwin, dIx, dIy) in shared memory, reduces the
// 2x2 normal matrix with warp REDUX, then iterates: bilinear taps of the next image, integer
// mismatch sums, warp reduce, float32 2x2 solve with cv2's exact termination rules.
// Integer sums are exact (int32 per lane, int64 across the warp) and converted to float32
// once; cv2 accumulates in float32 SIMD lanes, so positions agree to ~1e-3 px (tolerance
// 0.05 px) and status flags are identical.
#include "internal.cuh"

#define KLT_WARPS 4
#define W_BITS 14

struct KltArgs {
    const uint8_t* prev;
    const uint8_t* next;
    unsigned long long prev_stride, next_stride;
    unsigned long long off[VO_MAX_LEVELS];
    int w[VO_MAX_LEVELS], h[VO_MAX_LEVELS], pitch[VO_MAX_LEVELS];
    int levels;
    const VoSeqExt* ext;    // [batch] per-sequence level counts and level sizes, nullptr: levels / w / h above for every sequence
    int batch, n_fixed;
    // up to two point sets per sequence (landmark keypoints, candidate keypoints): [batch][cap[s]]
    int cap[2];
    const int* n_pts[2];
    const float* pts[2];
    float* out[2];
    uint8_t* status[2];
    float* err[2];
    int win_w, win_h, max_count;
    double eps_sq;
    float min_eig_thr;
    float min_eig_num;      // v3: minEig < min_eig_thr as a bound on minEig's numerator (min_eig_num_bound)
    float eps_lo, eps_hi;   // eps_sq * (1 -+ 1e-6) in float: outside this band the float test decides
    // shared-memory carve-up (bytes, per warp)
    int patch_stride, smem_patch, smem_der, smem_iwin, smem_di, smem_per_warp;
    int* queue;             // v3: [0] next feature slot, [1] warps that have found the queue empty (both 0 between launches)
};

__device__ __forceinline__ long long warp_sum_i64(int v)
{
    // exact 64-bit sum of 32 int32 lanes with two REDUX ops
    int lo = v & 0xFFFF;
    int hi = v >> 16;
    int slo = __reduce_add_sync(0xffffffffu, lo);
    int shi = __reduce_add_sync(0xffffffffu, hi);
    return (long long)shi * 65536ll + (long long)slo;
}

__device__ __forceinline__ int floor_to_int(float v)
{
    // cvFloor on x86: non-finite / out-of-range -> INT_MIN ("out of image")
    if (!(fabsf(v) < 1.0e9f)) return INT_MIN;
    return __float2int_rd(v);
}

__device__ __forceinline__ void bilinear_weights(float a, float b, int& w00, int& w01, int& w10, int& w11)
{
    const float s = (float)(1 << W_BITS);
    w00 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), __fsub_rn(1.f, b)), s));
    w01 = __float2int_rn(__fmul_rn(__fmul_rn(a, __fsub_rn(1.f, b)), s));
    w10 = __float2int_rn(__fmul_rn(__fmul_rn(__fsub_rn(1.f, a), b), s));
    w11 = (1 << W_BITS) - w00 - w01 - w10;
}

// EXT: the sequences have their own level counts and level sizes (a.ext); otherwise a.levels / a.w / a.h hold for all
template <int WW, int WH, bool EXT>
__global__ void __launch_bounds__(KLT_WARPS * 32)
klt_kernel(const KltArgs a)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    const long long gw = (long long)blockIdx.x * KLT_WARPS + warp;
    const int cap_all = a.cap[0] + a.cap[1];
    const int seq = (int)(gw / cap_all);
    int pi = (int)(gw - (long long)seq * cap_all);
    if (seq >= a.batch) return;
    const int seg = pi >= a.cap[0] ? 1 : 0;
    pi -= seg ? a.cap[0] : 0;
    const int n_here = a.n_pts[seg] ? a.n_pts[seg][seq] : a.n_fixed;
    if (pi >= n_here) return;

    const int ww = WW ? WW : a.win_w;
    const int wh = WH ? WH : a.win_h;
    const int wsz = ww * wh;
    uint8_t* wbase = smem + (size_t)warp * a.smem_per_warp;
    uint8_t* patch = wbase;                                              // (wh+3) rows x patch_stride
    int* der = reinterpret_cast<int*>(wbase + a.smem_patch);            // (wh+1) x (ww+1), Ix | Iy<<16
    short* Iwin = reinterpret_cast<short*>(wbase + a.smem_patch + a.smem_der);
    int* dI = reinterpret_cast<int*>(wbase + a.smem_patch + a.smem_der + a.smem_iwin);
    const int PS = a.patch_stride;

    const uint8_t* prev = a.prev + (size_t)seq * a.prev_stride;
    const uint8_t* next = a.next + (size_t)seq * a.next_stride;
    const size_t pidx = (size_t)seq * a.cap[seg] + pi;
    const float px0 = a.pts[seg][2 * pidx], py0 = a.pts[seg][2 * pidx + 1];
    const float hwx = (ww - 1) * 0.5f, hwy = (wh - 1) * 0.5f;
    const float FLT_SCALE = 1.f / (1 << 20);

    float outx = 0.f, outy = 0.f;
    int st = 1;
    float e = 0.f;
    const int levels = EXT ? a.ext[seq].levels : a.levels;

    for (int level = levels - 1; level >= 0; --level) {
        const int lw = EXT ? a.ext[seq].w[level] : a.w[level], lh = EXT ? a.ext[seq].h[level] : a.h[level];
        const int pitch = a.pitch[level];
        const uint8_t* I = prev + a.off[level];
        const uint8_t* J = next + a.off[level];
        const float sc = (float)(1.0 / (double)(1 << level));
        float ppx = __fmul_rn(px0, sc), ppy = __fmul_rn(py0, sc);
        float nx, ny;
        if (level == levels - 1) { nx = ppx; ny = ppy; }
        else { nx = __fmul_rn(outx, 2.f); ny = __fmul_rn(outy, 2.f); }
        outx = nx; outy = ny;
        ppx = __fsub_rn(ppx, hwx); ppy = __fsub_rn(ppy, hwy);
        const int ipx = floor_to_int(ppx), ipy = floor_to_int(ppy);
        if (ipx < -ww || ipx >= lw || ipy < -wh || ipy >= lh) {
            if (level == 0) { st = 0; e = 0.f; }
            continue;
        }
        int iw00, iw01, iw10, iw11;
        bilinear_weights(__fsub_rn(ppx, (float)ipx), __fsub_rn(ppy, (float)ipy), iw00, iw01, iw10, iw11);

        // ---- stage the (ww+3) x (wh+3) neighbourhood of I (origin ip-1) with 32-bit loads ----
        __syncwarp();
        const uint8_t* src0 = I + (long long)(ipy - 1) * pitch + (ipx - 1);
        const int mis = (int)(reinterpret_cast<uintptr_t>(src0) & 3);
        {
            const uint32_t* srcw = reinterpret_cast<const uint32_t*>(src0 - mis);
            const int wpr = (mis + ww + 3 + 3) >> 2;  // words per row
            const int nwords = wpr * (wh + 3);
            const int pw = pitch >> 2, psw = PS >> 2;
            uint32_t* pw32 = reinterpret_cast<uint32_t*>(patch);
            for (int k = lane; k < nwords; k += 32) {
                int r = k / wpr, c = k - r * wpr;
                pw32[r * psw + c] = __ldg(srcw + (long long)r * pw + c);
            }
        }
        __syncwarp();
        // patch(y, x) for y in [-1, wh+1], x in [-1, ww+1]  ->  patch[(y+1)*PS + mis + x + 1]
        const uint8_t* pc = patch + PS + mis + 1;

        // ---- Scharr derivative on the (ww+1) x (wh+1) tap grid, zero outside the image ----
        const int gw1 = ww + 1;
        const int ngrid = gw1 * (wh + 1);
        for (int k = lane; k < ngrid; k += 32) {
            int gy = k / gw1, gx = k - gy * gw1;
            int X = ipx + gx, Y = ipy + gy;
            int val = 0;
            if (X >= 0 && X < lw && Y >= 0 && Y < lh) {
                const uint8_t* c = pc + gy * PS + gx;
                int p00 = c[-PS - 1], p01 = c[-PS], p02 = c[-PS + 1];
                int p10 = c[-1], p12 = c[1];
                int p20 = c[PS - 1], p21 = c[PS], p22 = c[PS + 1];
                int ix = ((p02 + p22) * 3 + p12 * 10) - ((p00 + p20) * 3 + p10 * 10);
                int iy = ((p22 - p02) + (p20 - p00)) * 3 + (p21 - p01) * 10;
                val = (ix & 0xFFFF) | (iy << 16);
            }
            der[k] = val;
        }
        __syncwarp();

        // ---- template: Iwin, dIx, dIy and the normal matrix ----
        int sA11 = 0, sA12 = 0, sA22 = 0;
        for (int k = lane; k < wsz; k += 32) {
            int y = k / ww, x = k - y * ww;
            const uint8_t* c = pc + y * PS + x;
            int iv = (c[0] * iw00 + c[1] * iw01 + c[PS] * iw10 + c[PS + 1] * iw11 + (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5);
            const int* d = der + y * gw1 + x;
            int d00 = d[0], d01 = d[1], d10 = d[gw1], d11 = d[gw1 + 1];
            int ixv = ((short)d00 * iw00 + (short)d01 * iw01 + (short)d10 * iw10 + (short)d11 * iw11 + (1 << (W_BITS - 1))) >> W_BITS;
            int iyv = ((d00 >> 16) * iw00 + (d01 >> 16) * iw01 + (d10 >> 16) * iw10 + (d11 >> 16) * iw11 + (1 << (W_BITS - 1))) >> W_BITS;
            Iwin[k] = (short)iv;
            dI[k] = (ixv & 0xFFFF) | (iyv << 16);
            sA11 += ixv * ixv;
            sA12 += ixv * iyv;
            sA22 += iyv * iyv;
        }
        const float A11 = __fmul_rn(__ll2float_rn(warp_sum_i64(sA11)), FLT_SCALE);
        const float A12 = __fmul_rn(__ll2float_rn(warp_sum_i64(sA12)), FLT_SCALE);
        const float A22 = __fmul_rn(__ll2float_rn(warp_sum_i64(sA22)), FLT_SCALE);
        float D = __fsub_rn(__fmul_rn(A11, A22), __fmul_rn(A12, A12));
        const float dA = __fsub_rn(A11, A22);
        const float minEig = __fdiv_rn(
            __fsub_rn(__fadd_rn(A22, A11),
                      __fsqrt_rn(__fadd_rn(__fmul_rn(dA, dA), __fmul_rn(__fmul_rn(4.f, A12), A12)))),
            (float)(2 * ww * wh));
        if (minEig < a.min_eig_thr || D < 1.192092896e-07f) {
            if (level == 0) st = 0;
            continue;
        }
        D = __fdiv_rn(1.f, D);
        nx = __fsub_rn(nx, hwx); ny = __fsub_rn(ny, hwy);
        float pdx = 0.f, pdy = 0.f;
        __syncwarp();

        for (int j = 0; j < a.max_count; ++j) {
            const int inx = floor_to_int(nx), iny = floor_to_int(ny);
            if (inx < -ww || inx >= lw || iny < -wh || iny >= lh) {
                if (level == 0) st = 0;
                break;
            }
            bilinear_weights(__fsub_rn(nx, (float)inx), __fsub_rn(ny, (float)iny), iw00, iw01, iw10, iw11);
            const uint8_t* Jp = J + (long long)iny * pitch + inx;
            int sb1 = 0, sb2 = 0;
            for (int k = lane; k < wsz; k += 32) {
                int y = k / ww, x = k - y * ww;
                const uint8_t* c = Jp + y * pitch + x;
                int diff = ((__ldg(c) * iw00 + __ldg(c + 1) * iw01 + __ldg(c + pitch) * iw10 + __ldg(c + pitch + 1) * iw11 +
                             (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5)) - Iwin[k];
                int d = dI[k];
                sb1 += diff * (short)d;
                sb2 += diff * (d >> 16);
            }
            const float b1 = __fmul_rn(__ll2float_rn(warp_sum_i64(sb1)), FLT_SCALE);
            const float b2 = __fmul_rn(__ll2float_rn(warp_sum_i64(sb2)), FLT_SCALE);
            const float dx = __fmul_rn(__fsub_rn(__fmul_rn(A12, b2), __fmul_rn(A22, b1)), D);
            const float dy = __fmul_rn(__fsub_rn(__fmul_rn(A12, b1), __fmul_rn(A11, b2)), D);
            nx = __fadd_rn(nx, dx); ny = __fadd_rn(ny, dy);
            outx = __fadd_rn(nx, hwx); outy = __fadd_rn(ny, hwy);
            if (__dadd_rn(__dmul_rn((double)dx, (double)dx), __dmul_rn((double)dy, (double)dy)) <= a.eps_sq) break;
            if (j > 0 && fabsf(__fadd_rn(dx, pdx)) < 0.01f && fabsf(__fadd_rn(dy, pdy)) < 0.01f) {
                outx = __fsub_rn(outx, __fmul_rn(dx, 0.5f));
                outy = __fsub_rn(outy, __fmul_rn(dy, 0.5f));
                break;
            }
            pdx = dx; pdy = dy;
        }

        if (st && level == 0) {
            const float qx = __fsub_rn(outx, hwx), qy = __fsub_rn(outy, hwy);
            const int inx = floor_to_int(qx), iny = floor_to_int(qy);
            if (inx < -ww || inx >= lw || iny < -wh || iny >= lh) {
                st = 0;
                continue;
            }
            bilinear_weights(__fsub_rn(qx, (float)inx), __fsub_rn(qy, (float)iny), iw00, iw01, iw10, iw11);
            const uint8_t* Jp = J + (long long)iny * pitch + inx;
            int se = 0;
            for (int k = lane; k < wsz; k += 32) {
                int y = k / ww, x = k - y * ww;
                const uint8_t* c = Jp + y * pitch + x;
                int diff = ((__ldg(c) * iw00 + __ldg(c + 1) * iw01 + __ldg(c + pitch) * iw10 + __ldg(c + pitch + 1) * iw11 +
                             (1 << (W_BITS - 5 - 1))) >> (W_BITS - 5)) - Iwin[k];
                se += abs(diff);
            }
            e = __fdiv_rn(__ll2float_rn(warp_sum_i64(se)), (float)(32 * ww * wh));
        }
    }
    if (lane == 0) {
        a.out[seg][2 * pidx] = outx;
        a.out[seg][2 * pidx + 1] = outy;
        a.status[seg][pidx] = (uint8_t)st;
        if (a.err[seg]) a.err[seg][pidx] = e;
    }
}

#include "klt_v3.cuh"

#define KLT_QUEUE_SLOTS 1024
#define KLT_QUEUE_INTS 8   // one 32-byte sector per slot

int vo_klt_launch2(b200vo_ctx* ctx, const PyrGeom& g, const uint8_t* d_prev_slab, size_t prev_stride,
                   const uint8_t* d_next_slab, size_t next_stride, int batch, const KltPointSet* sets, int n_sets,
                   int n_fixed, const KltParams& kp, cudaStream_t stream, const VoSeqExt* d_ext)
{
    if (batch <= 0 || n_sets <= 0) return 0;
    KltArgs a{};
    a.prev = d_prev_slab; a.next = d_next_slab;
    a.prev_stride = prev_stride; a.next_stride = next_stride;
    a.levels = g.levels;
    for (int l = 0; l < g.levels; ++l) {
        a.off[l] = g.off[l]; a.w[l] = g.w[l]; a.h[l] = g.h[l]; a.pitch[l] = g.pitch[l];
    }
    a.ext = d_ext;
    a.batch = batch; a.n_fixed = n_fixed;
    for (int s = 0; s < 2; ++s) {
        const bool on = s < n_sets;
        a.cap[s] = on ? sets[s].cap : 0;
        a.n_pts[s] = on ? sets[s].n : nullptr;
        a.pts[s] = on ? sets[s].pts : nullptr;
        a.out[s] = on ? sets[s].out : nullptr;
        a.status[s] = on ? sets[s].status : nullptr;
        a.err[s] = on ? sets[s].err : nullptr;
    }
    if (a.cap[0] + a.cap[1] <= 0) return 0;
    a.win_w = kp.win_w; a.win_h = kp.win_h; a.max_count = kp.max_count;
    a.eps_sq = kp.eps_sq; a.min_eig_thr = kp.min_eig_thr;
    a.eps_lo = (float)(kp.eps_sq * (1.0 - 1e-6)); a.eps_hi = (float)(kp.eps_sq * (1.0 + 1e-6));
    a.patch_stride = (int)vo_align((size_t)kp.win_w + 3 + 3, 4);
    a.smem_patch = (int)vo_align((size_t)a.patch_stride * (kp.win_h + 3), 16);
    a.smem_der = (int)vo_align((size_t)(kp.win_w + 1) * (kp.win_h + 1) * 4, 16);
    a.smem_iwin = (int)vo_align((size_t)kp.win_w * kp.win_h * 2, 16);
    a.smem_di = (int)vo_align((size_t)kp.win_w * kp.win_h * 4, 16);
    a.smem_per_warp = a.smem_patch + a.smem_der + a.smem_iwin + a.smem_di;
    size_t smem = (size_t)a.smem_per_warp * KLT_WARPS;
    const long long total_warps = (long long)batch * (a.cap[0] + a.cap[1]);
    const unsigned grid = (unsigned)((total_warps + KLT_WARPS - 1) / KLT_WARPS);
    void (*kern)(const KltArgs) = d_ext ? klt_kernel<0, 0, true> : klt_kernel<0, 0, false>;
    bool staged = false;
    // the staged kernel (persistent warps + work queue) for the two window sizes it is built for; the queue counter is
    // an int, so a launch of 2^30 features or more takes the generic kernel (same arithmetic, same results), and so do
    // frames of 2^22 pixels or more in a dimension (the staged kernel's floor is exact below that: floor_v3)
    const bool sized = (kp.win_w == 21 && kp.win_h == 21) || (kp.win_w == 15 && kp.win_h == 15);
    unsigned launch_grid = grid;
    if (sized && total_warps < (1ll << 30) && g.w[0] < (1 << 22) && g.h[0] < (1 << 22)) {
        int min_ctas;
        staged = true;
        a.min_eig_num = min_eig_num_bound(kp.min_eig_thr, (float)(2 * kp.win_w * kp.win_h));
        // per-sequence extents: the instances that read them (a uniform batch keeps the ones that take the launch's geometry)
        if (kp.win_w == 21) {
            kern = d_ext ? klt_kernel_v3<21, 21, true> : klt_kernel_v3<21, 21, false>;
            smem = (size_t)KV3<21, 21>::PER_WARP * KLT_WARPS + 64; min_ctas = KV3<21, 21>::MIN_CTAS;
        } else {
            kern = d_ext ? klt_kernel_v3<15, 15, true> : klt_kernel_v3<15, 15, false>;
            smem = (size_t)KV3<15, 15>::PER_WARP * KLT_WARPS + 64; min_ctas = KV3<15, 15>::MIN_CTAS;
        }
        if (!ctx->d_klt_queue.p) {
            VO_TRY(vo_reserve(ctx, ctx->d_klt_queue, (size_t)KLT_QUEUE_SLOTS * KLT_QUEUE_INTS * sizeof(int)));
            VO_CUDA(ctx, cudaMemsetAsync(ctx->d_klt_queue.p, 0, (size_t)KLT_QUEUE_SLOTS * KLT_QUEUE_INTS * sizeof(int), stream));
            VO_CUDA(ctx, cudaStreamSynchronize(stream));   // other streams of this context launch trackers too
        }
        // a ring of counters: launches that run concurrently (landmark / candidate sets, chunk streams) never share one,
        // and each kernel re-arms its own slot when its last warp retires
        a.queue = (int*)ctx->d_klt_queue.p + (size_t)(ctx->klt_queue_next++ % KLT_QUEUE_SLOTS) * KLT_QUEUE_INTS;
        const unsigned resident = (unsigned)(ctx->num_sms * min_ctas);
        launch_grid = grid < resident ? grid : resident;
    }
    {   // function attributes: once per kernel and process (the calls cost microseconds each on the launch path)
        static void* configured[8] = {};
        bool seen = false;
        int free_slot = -1;
        for (int i = 0; i < 8; ++i) { seen = seen || configured[i] == (void*)kern; if (!configured[i] && free_slot < 0) free_slot = i; }
        if (!seen) {
            if (smem > 48 * 1024)
                VO_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            if (staged)   // the staged kernels live in shared memory: let 8 CTAs (64 registers each) fit
                VO_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
            if (free_slot >= 0 && staged) configured[free_slot] = (void*)kern;   // the generic kernel's smem size varies per call
        }
    }
    kern<<<launch_grid, KLT_WARPS * 32, smem, stream>>>(a);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// trace aid (B200VO_TRACE_FILE): (first feature claimed, last warp retired) GPU wall-clock pairs of every queue slot
void vo_klt_trace_read(b200vo_ctx* ctx, std::vector<unsigned long long>& out)
{
    out.clear();
    if (!ctx->d_klt_queue.p) return;
    std::vector<unsigned long long> raw((size_t)KLT_QUEUE_SLOTS * KLT_QUEUE_INTS / 2);
    if (cudaMemcpy(raw.data(), ctx->d_klt_queue.p, raw.size() * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return;
    for (int s = 0; s < KLT_QUEUE_SLOTS; ++s) { out.push_back(raw[(size_t)s * 4 + 1]); out.push_back(raw[(size_t)s * 4 + 2]); }
}
