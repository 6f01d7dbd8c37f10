// P3P-RANSAC on the GPU (replaces cv2.solvePnPRansac(..., flags=SOLVEPNP_P3P) at reference
// VisualOdometryPipeLine.py:343; spec SURVEY.md A.6-A.8 and oracle/pnp_oracle.c header).
//
// All `iters` hypotheses are drawn, solved and scored at once; a sequential replay of the
// per-hypothesis inlier counts then reproduces OpenCV's "first strictly better model wins,
// shrink niters" loop, so the winner (and therefore the inlier mask) is the one cv2 returns.
//   1. ransac_samples_kernel<4> (ransac.cuh) bit-exact cv::RNG((uint64)-1) 4-subsets (raw stream table + parallel mod)
//   2. pnp_solve_kernel     one thread per hypothesis: FP64 P3P + 4-point disambiguation
//   3. pnp_score_kernel     (point tile x hypothesis tile): FP64 projection -> f32 error,
//                           warp-aggregated inlier counts (ballot+popc, one atomicAdd per warp)
//   4. pnp_select_kernel    replay + winner mask + ordered inlier compaction
//   5. pnp_epnp_kernel      EPnP refit on the inliers (block reductions + small FP64 solves)
// Every kernel is batched over independent sequences (blockIdx.z / blockIdx.x = sequence).
#include "internal.cuh"
#include "mathdev.cuh"
#include "pnp.cuh"
#include "ransac.cuh"

using namespace vo;

// One of the four camera doubles (fx, fy, cx, cy) of a sequence, read where it is used: the loads are not merged or hoisted,
// so no register holds the camera across the solvers' long live ranges (the fused kernel is at its register limit)
__device__ __forceinline__ double cam_at(const double* cam, int k) { return ((const volatile double*)cam)[k]; }

// ------------------------------------------------------------------------------------------
// 2. minimal solver: one thread per hypothesis
// ------------------------------------------------------------------------------------------
// One hypothesis: P3P on the first 3 points of the sample, the 4th picks the candidate.  Writes R|t (re-expanded
// from rvec, as PnPRansacCallback stores its model) to h[12] and rvec to hr[3]; returns 0 when there is no model.
// cam = the sequence's fx, fy, cx, cy.
__device__ inline int pnp_solve_one(const double* cam, const float* obj, const float* img, const int* smp, double* h, double* hr)
{
    double X[12], xn[8], uv[8];
    const double ifx = 1. / cam_at(cam, 0), ify = 1. / cam_at(cam, 1);
    for (int k = 0; k < 4; ++k) {
        const int s = smp[k];
        X[3 * k] = obj[3 * s]; X[3 * k + 1] = obj[3 * s + 1]; X[3 * k + 2] = obj[3 * s + 2];
        uv[2 * k] = img[2 * s]; uv[2 * k + 1] = img[2 * s + 1];
        // cv2 normalises with undistortPoints on CV_32F input: double arithmetic, float32 result
        xn[2 * k] = (double)(float)((uv[2 * k] - cam_at(cam, 2)) * ifx);
        xn[2 * k + 1] = (double)(float)((uv[2 * k + 1] - cam_at(cam, 3)) * ify);
    }
    double R[4][9], t[4][3];
    const int ns = p3p(X, xn, R, t);
    int best = -1;
    double best_e = 0;
    for (int s = 0; s < ns; ++s) {
        double e = 0;
        for (int k = 0; k < 4; ++k) {
            double u, v;
            project_pt(R[s], t[s], cam_at(cam, 0), cam_at(cam, 1), cam_at(cam, 2), cam_at(cam, 3), X[3 * k], X[3 * k + 1], X[3 * k + 2], u, v);
            const double dx = uv[2 * k] - u, dy = uv[2 * k + 1] - v;
            e += dx * dx + dy * dy;
        }
        if (!isfinite(e)) continue;
        if (best < 0 || e < best_e) { best = s; best_e = e; }
    }
    if (best < 0) return 0;
    // the model is stored as rvec|tvec and re-expanded for scoring (as PnPRansacCallback does)
    double rv[3], Rr[9];
    R_to_rodrigues(R[best], rv);
    rodrigues_to_R(rv, Rr);
    for (int k = 0; k < 9; ++k) h[k] = Rr[k];
    for (int k = 0; k < 3; ++k) h[9 + k] = t[best][k];
    hr[0] = rv[0]; hr[1] = rv[1]; hr[2] = rv[2];
    return 1;
}

__global__ void __launch_bounds__(64)
pnp_solve_kernel(PnpArgs a)
{
    const int b = blockIdx.y;
    const int it = a.h_begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= a.h_end) return;
    if (!a.head && it >= a.need[b]) return;      // the sequential loop can no longer reach this hypothesis
    const size_t hidx = (size_t)b * a.iters + it;
    a.counts[hidx] = 0;
    a.hyp_ok[hidx] = 0;
    const int* smp = a.samples + hidx * 4;
    const int N = a.n[b];
    if (smp[0] < 0 || N < 4) return;
    a.hyp_ok[hidx] = pnp_solve_one(&a.intr[b].fx, a.obj + (size_t)b * a.cap * 3, a.img + (size_t)b * a.cap * 2, smp, a.hyp + hidx * 12,
                                   a.hyp_rvec + hidx * 3);
}

// ------------------------------------------------------------------------------------------
// 3. scoring
// ------------------------------------------------------------------------------------------
#define SCORE_HT 32   // hypotheses per block
#define PNP_HEAD 32   // hypotheses solved and scored before the first look at the adaptive stop

__device__ __forceinline__ bool pnp_is_inlier(const double* h, double fx, double fy, double cx, double cy,
                                              double X, double Y, double Z, float iu, float iv, float thr_sq)
{
    double u, v;
    project_pt(h, h + 9, fx, fy, cx, cy, X, Y, Z, u, v);
    const float pu = (float)u, pv = (float)v;      // projectPoints output is float32
    const float dx = __fsub_rn(iu, pu), dy = __fsub_rn(iv, pv);
    const float e = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    return e <= thr_sq;                              // NaN compares false
}

// Head chunk bookkeeping: the LAST CTA of a sequence to finish (ticket counter, no waiting) replays
// cv2's loop over the head hypotheses; what it leaves in `niters` bounds every later replay, so
// the tail launches skip hypotheses >= need[b] (typically all of them: at 10 % outliers cv2 itself
// stops after ~5 iterations).
__device__ __forceinline__ void pnp_head_done(const PnpArgs& a, int b, int N)
{
    __shared__ int s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(a.ticket + b, 1) == (int)(gridDim.x * gridDim.y) - 1;
    }
    __syncthreads();
    if (!s_last || threadIdx.x != 0) return;
    __threadfence();
    int niters = a.iters > 1 ? a.iters : 1;
    if (N == 4) niters = 1;
    else if (N > 4) {
        const size_t hb = (size_t)b * a.iters;
        int max_good = 0;
        for (int it = a.h_begin; it < a.h_end && it < niters; ++it) {
            if (!((volatile int*)a.hyp_ok)[hb + it]) continue;
            const int good = ((volatile int*)a.counts)[hb + it];
            if (good > (max_good > 3 ? max_good : 3)) {
                max_good = good;
                niters = ransac_update_num_iters(a.conf, (double)(N - good) / N, 4, niters);
            }
        }
    } else niters = 0;
    a.need[b] = niters;
}

__global__ void __launch_bounds__(256)
pnp_score_kernel(PnpArgs a)
{
    __shared__ double s_h[SCORE_HT * 12];
    __shared__ int s_ok[SCORE_HT];
    const int b = blockIdx.z;
    const int N = a.n[b];
    const int p0 = blockIdx.x * blockDim.x;
    const int h0 = a.h_begin + blockIdx.y * SCORE_HT;
    if (!a.head && (p0 >= N || N <= 4 || h0 >= a.need[b])) return;
    if (a.head && (p0 >= N || N <= 4)) { pnp_head_done(a, b, N); return; }
    const int nh = min(SCORE_HT, a.h_end - h0);
    const size_t hbase = (size_t)b * a.iters + h0;
    for (int k = threadIdx.x; k < nh * 12; k += blockDim.x) s_h[k] = a.hyp[hbase * 12 + k];
    if (threadIdx.x < nh) s_ok[threadIdx.x] = a.hyp_ok[hbase + threadIdx.x];
    __syncthreads();
    const int i = p0 + threadIdx.x;
    const bool live = i < N;
    double X = 0, Y = 0, Z = 0;
    float iu = 0, iv = 0;
    if (live) {
        const float* o = a.obj + ((size_t)b * a.cap + i) * 3;
        const float* m = a.img + ((size_t)b * a.cap + i) * 2;
        X = o[0]; Y = o[1]; Z = o[2];
        iu = m[0]; iv = m[1];
    }
    const int lane = threadIdx.x & 31;
    const VoIntrinsics& cam = a.intr[b];
    const double fx = cam.fx, fy = cam.fy, cx = cam.cx, cy = cam.cy;
    for (int h = 0; h < nh; ++h) {
        if (!s_ok[h]) continue;   // block-uniform
        const bool in = live && pnp_is_inlier(s_h + h * 12, fx, fy, cx, cy, X, Y, Z, iu, iv, a.thr_sq);
        const unsigned m = __ballot_sync(0xffffffffu, in);
        if (lane == 0 && m) atomicAdd(a.counts + hbase + h, __popc(m));
    }
    if (a.head) pnp_head_done(a, b, N);
}

// ------------------------------------------------------------------------------------------
// 4. select: replay cv2's sequential loop, then winner mask + ordered compaction
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pnp_select_kernel(PnpArgs a)
{
    __shared__ int s_win, s_run;
    __shared__ double s_h[12];
    const int b = blockIdx.x;
    const int N = a.n[b];
    const size_t hb = (size_t)b * a.iters;
    if (threadIdx.x == 0) {
        int win = -1, run = 0;
        if (N == 4) { win = a.hyp_ok[hb] ? 0 : -1; run = 1; }
        else if (N > 4) {
            int niters = a.iters > 1 ? a.iters : 1, max_good = 0, it;
            for (it = 0; it < niters; ++it) {
                if (!a.hyp_ok[hb + it]) continue;
                const int good = a.counts[hb + it];
                if (good > (max_good > 3 ? max_good : 3)) {
                    win = it; max_good = good;
                    niters = ransac_update_num_iters(a.conf, (double)(N - good) / N, 4, niters);
                }
            }
            run = it;
        }
        s_win = win; s_run = run;
    }
    __syncthreads();
    const int win = s_win;
    uint8_t* mask = a.mask + (size_t)b * a.cap;
    int* inl = a.inliers + (size_t)b * a.cap;
    if (threadIdx.x == 0) { a.winner[b] = win; a.iters_run[b] = s_run; }
    if (win < 0) {
        for (int i = threadIdx.x; i < a.cap; i += blockDim.x) mask[i] = 0;
        if (threadIdx.x == 0) { a.n_inliers[b] = 0; a.ok[b] = 0; }
        return;
    }
    if (threadIdx.x < 12) s_h[threadIdx.x] = a.hyp[(hb + win) * 12 + threadIdx.x];
    __syncthreads();
    // over every slot, so that keep() writes the whole mask
    const int M = cta_compact<256>(a.cap, [&](int i) {
        bool in = false;
        if (i < N) {
            if (N == 4) in = true;
            else {
                const float* o = a.obj + ((size_t)b * a.cap + i) * 3;
                const float* m = a.img + ((size_t)b * a.cap + i) * 2;
                in = pnp_is_inlier(s_h, a.intr[b].fx, a.intr[b].fy, a.intr[b].cx, a.intr[b].cy, o[0], o[1], o[2], m[0], m[1], a.thr_sq);
            }
        }
        mask[i] = in ? 1 : 0;
        return in;
    }, [&](int i, int o) { inl[o] = i; });
    if (threadIdx.x == 0) {
        a.n_inliers[b] = M;
        a.ok[b] = 1;
        // RANSAC model (what cv2 falls back to / returns for N == 4)
        double* pose = a.pose + (size_t)b * 6;
        const double* hr = a.hyp_rvec + (hb + win) * 3;
        pose[0] = hr[0]; pose[1] = hr[1]; pose[2] = hr[2];
        pose[3] = s_h[9]; pose[4] = s_h[10]; pose[5] = s_h[11];
    }
}

// ------------------------------------------------------------------------------------------
// 5. EPnP refit on the inliers (SURVEY A.8; OpenCV epnp.cpp algorithm, float64 inputs)
// ------------------------------------------------------------------------------------------
// optional phase stamps (clock64 of thread 0) for benchmarks/pose_phases.py: PnpArgs::phase_clk, [batch][16]
__device__ __forceinline__ void phase_stamp(const PnpArgs& a, int b, int k)
{
    if (a.phase_clk && threadIdx.x == 0) {
        a.phase_clk[(size_t)b * 16 + k] = clock64();
        if (k == 0 || k == 8) {   // wall-clock stamps + SM id: where the CTA ran beside the tracker (B200VO_TRACE_FILE)
            unsigned long long t; unsigned sm;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
            asm volatile("mov.u32 %0, %smid;" : "=r"(sm));
            a.phase_clk[(size_t)b * 16 + (k == 0 ? 12 : 14)] = (long long)t;
            a.phase_clk[(size_t)b * 16 + 13] = sm;
        }
    }
}

#define EPNP_T 256
#define EPNP_JT 160   // threads of the block that take part in the 12x12 eigen-decomposition (144 elements, 5 warps)

__device__ __forceinline__ void bar_jacobi() { asm volatile("bar.sync 1, %0;" ::"n"(EPNP_JT) : "memory"); }

// 1/x to ~1 ulp without the IEEE division routine: hardware seed (2^-23) + two Newton steps
__device__ __forceinline__ double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    r = fma(r, fma(-x, r, 1.0), r);
    r = fma(r, fma(-x, r, 1.0), r);
    return r;
}

struct EpnpShared {
    double red[8 * 56];
    double out[56];
    double cws[4][3];
    double ci[9];       // inverse of the control-point basis
    double v4[4][12];   // eigenvectors of MtM for the 4 smallest eigenvalues, smallest first
    double L[60], rho[6];
    double Rs[3][9], ts[3][3];
    double mom_aX[12];  // sum_i alpha_ij X_ik
    double mom_a[4];    // sum_i alpha_ij
    double alpha0[4];   // barycentric coords of the first inlier (solve_for_sign)
    double jac[2][288]; // double-buffered [A (12x12) | V (12x12)]
    double rc[EPNP_JT / 32][12], rs[EPNP_JT / 32][12];   // per warp: this round's rotation seen from index k: x_k' = rc[k] x_k + rs[k] x_partner(k)
    unsigned char partner[11 * 12];
};

// Symmetric 12x12 eigen-decomposition by two-sided Jacobi rotations with the round-robin (tournament) ordering:
// 11 rounds per sweep, 6 disjoint (p,q) pairs per round.  One thread per matrix element: A' = J^T A J and V' = V J
// are each ONE read-compute-write pass per round (the old form needed a column pass, a row pass and three warp
// barriers on one warp), double-buffered so that a round costs ONE block barrier: every warp computes the round's six
// rotations for itself (lanes 0-5, a warp-private copy in shared memory, __syncwarp) instead of waiting for one warp
// to publish them.  The rotation is the small-angle solution in half-angle form,
//     c = sqrt((1 + |d|/h) / 2),  s = sgn(d) b / (2 h c),   d = a_qq - a_pp, b = 2 a_pq, h = sqrt(d^2 + b^2),
// i.e. two reciprocal square roots and no division (1 + |d|/h never cancels).
// Called by threads [0, EPNP_JT); S.jac[0][0..143] holds A on entry.  Returns the buffer index holding the result
// (A's diagonal = eigenvalues, V's columns = eigenvectors).  Only used for EPnP's M^T M, where the result is
// independent of eigenvector signs and of the rotation order (unlike the 3x3 control-point SVD, which replays
// OpenCV's order exactly).
__device__ inline int block_jacobi_eig12(EpnpShared& S, int tid)
{
    const bool act = tid < 144;
    const int i = act ? tid / 12 : 0, j = act ? tid - 12 * i : 0;
    const int lane = tid & 31, warp = tid >> 5;
    double* rc = S.rc[warp];
    double* rs = S.rs[warp];
    if (act) S.jac[0][144 + tid] = (i == j) ? 1.0 : 0.0;
    int cur = 0;
    bar_jacobi();
    for (int sweep = 0; sweep < 30; ++sweep) {
        {   // convergence: squared off-diagonal mass relative to the diagonal (every warp for itself: no barrier)
            const double* A = S.jac[cur];
            double off = 0, dia = 0;
            for (int k = lane; k < 144; k += 32) {
                const double v = A[k];
                if (k / 12 == k % 12) dia += v * v; else off += v * v;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { off += __shfl_xor_sync(0xffffffffu, off, o); dia += __shfl_xor_sync(0xffffffffu, dia, o); }
            if (off <= 1e-30 * dia || off == 0) return cur;     // same value in every warp: uniform exit
        }
        for (int rnd = 0; rnd < 11; ++rnd) {
            const double* A = S.jac[cur];
            if (lane < 6) {
                int p = lane == 0 ? 11 : (rnd + lane) % 11;
                int q = (rnd + 11 - lane) % 11;
                if (p > q) { const int t = p; p = q; q = t; }
                const double apq = A[p * 12 + q];
                double c = 1.0, sn = 0.0;
                const double d = A[q * 12 + q] - A[p * 12 + p], b2 = 2 * apq;
                const double hh = d * d + b2 * b2;
                if (fabs(apq) > 1e-300 && hh > 1e-30 && hh < 1e30) {
                    const double rh = rsqrt_fast(hh);
                    const double u = fma(0.5 * fabs(d), rh, 0.5);        // (1 + |d|/h) / 2 in [0.5, 1]
                    const double ru = rsqrt_fast(u);
                    c = u * ru;
                    sn = (d >= 0 ? 0.5 : -0.5) * b2 * rh * ru;
                } else if (fabs(apq) > 1e-300) {                         // outside the float range of the seed: the slow exact form
                    const double theta = d / b2;
                    const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1));
                    c = 1 / sqrt(t * t + 1); sn = t * c;
                }
                if (!isfinite(c) || !isfinite(sn)) { c = 1.0; sn = 0.0; }
                rc[p] = c; rs[p] = -sn;     // x_p' = c x_p - s x_q
                rc[q] = c; rs[q] = sn;      // x_q' = s x_p + c x_q
            }
            __syncwarp();
            if (act) {
                const int pi = S.partner[rnd * 12 + i], pj = S.partner[rnd * 12 + j];
                const double ci_ = rc[i], si_ = rs[i], cj = rc[j], sj = rs[j];
                const double b_ij = cj * A[i * 12 + j] + sj * A[i * 12 + pj];        // (A J)[i][j]
                const double b_pj = cj * A[pi * 12 + j] + sj * A[pi * 12 + pj];      // (A J)[partner(i)][j]
                double* Nx = S.jac[cur ^ 1];
                Nx[i * 12 + j] = ci_ * b_ij + si_ * b_pj;                             // (J^T A J)[i][j]
                Nx[144 + i * 12 + j] = cj * A[144 + i * 12 + j] + sj * A[144 + i * 12 + pj];
            }
            bar_jacobi();
            cur ^= 1;
        }
    }
    return cur;
}

template <int NV>
__device__ __forceinline__ void block_reduce_sum(double* v, double* s_red /* [8][NV] */, double* s_out /* [NV] */)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) s_red[warp * NV + k] = x;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double x = 0;
        for (int w = 0; w < EPNP_T / 32; ++w) x += s_red[w * NV + threadIdx.x];
        s_out[threadIdx.x] = x;
    }
    __syncthreads();
}

__device__ inline void epnp_pose_from_betas(EpnpShared& S, const double* betas, double n, const double* Xbar, double* R, double* t)
{
    double ccs[4][3];
    for (int i = 0; i < 4; ++i)
        for (int k = 0; k < 3; ++k) {
            double s = 0;
            for (int j = 0; j < 4; ++j) s += betas[j] * S.v4[j][3 * i + k];
            ccs[i][k] = s;
        }
    // solve_for_sign: z of the first point in the camera frame
    const double z0 = S.alpha0[0] * ccs[0][2] + S.alpha0[1] * ccs[1][2] + S.alpha0[2] * ccs[2][2] + S.alpha0[3] * ccs[3][2];
    if (z0 < 0)
        for (int i = 0; i < 4; ++i) for (int k = 0; k < 3; ++k) ccs[i][k] = -ccs[i][k];
    // pc_i = sum_j alpha_ij ccs_j is linear in alpha: the centroid and the cross-covariance follow
    // from the moments sum alpha, sum alpha X^T gathered in the reduction pass.
    double pc0[3];
    for (int k = 0; k < 3; ++k)
        pc0[k] = (S.mom_a[0] * ccs[0][k] + S.mom_a[1] * ccs[1][k] + S.mom_a[2] * ccs[2][k] + S.mom_a[3] * ccs[3][k]) / n;
    double abt[9];
    for (int j = 0; j < 3; ++j)
        for (int k = 0; k < 3; ++k) {
            double s = 0;
            for (int q = 0; q < 4; ++q) s += ccs[q][j] * S.mom_aX[3 * q + k];
            abt[3 * j + k] = s - n * pc0[j] * Xbar[k];
        }
    double W[3], U[9], Vt[9], At[9];
    jacobi_svd<3>(abt, W, U, Vt, At);
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[3 * i + j] = U[3 * i] * Vt[j] + U[3 * i + 1] * Vt[3 + j] + U[3 * i + 2] * Vt[6 + j];
    if (det3(R) < 0) { R[6] = -R[6]; R[7] = -R[7]; R[8] = -R[8]; }
    for (int k = 0; k < 3; ++k) t[k] = pc0[k] - (R[3 * k] * Xbar[0] + R[3 * k + 1] * Xbar[1] + R[3 * k + 2] * Xbar[2]);
}

__device__ inline void epnp_gauss_newton(const double* L, const double* rho, double* b)
{
#pragma unroll 1
    for (int it = 0; it < 5; ++it) {
        double A[24], B[6], x[4];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const double* r = L + 10 * i;
            A[4 * i + 0] = 2 * r[0] * b[0] + r[1] * b[1] + r[3] * b[2] + r[6] * b[3];
            A[4 * i + 1] = r[1] * b[0] + 2 * r[2] * b[1] + r[4] * b[2] + r[7] * b[3];
            A[4 * i + 2] = r[3] * b[0] + r[4] * b[1] + 2 * r[5] * b[2] + r[8] * b[3];
            A[4 * i + 3] = r[6] * b[0] + r[7] * b[1] + r[8] * b[2] + 2 * r[9] * b[3];
            B[i] = rho[i] - (r[0] * b[0] * b[0] + r[1] * b[0] * b[1] + r[2] * b[1] * b[1] + r[3] * b[0] * b[2] +
                             r[4] * b[1] * b[2] + r[5] * b[2] * b[2] + r[6] * b[0] * b[3] + r[7] * b[1] * b[3] +
                             r[8] * b[2] * b[3] + r[9] * b[3] * b[3]);
        }
        qr_lstsq6<4>(A, B, x);
#pragma unroll
        for (int k = 0; k < 4; ++k) b[k] += x[k];
    }
}

// The refit, executed by one CTA of EPNP_T threads (every thread must call it; S is the CTA's scratch):
// obj/img are this sequence's correspondences, inl[0..M) the inlier indices, pose_out receives rvec|tvec
// (left untouched when the result is not finite -- the caller has put the RANSAC model there); cam = fx, fy, cx, cy.
__device__ inline void epnp_block(const PnpArgs& a, const double* cam, EpnpShared& S, const float* obj, const float* img, const int* inl, int M,
                                  double* pose_out, int b)
{
    const int tid = threadIdx.x;
    const double n = (double)M;
    const double ifx = 1. / cam_at(cam, 0), ify = 1. / cam_at(cam, 1);
    // tournament partner table (built here, consumed after several barriers)
    for (int k = tid; k < 66; k += EPNP_T) {
        const int rnd = k / 6, pr = k - rnd * 6;
        const int p = pr == 0 ? 11 : (rnd + pr) % 11, q = (rnd + 11 - pr) % 11;
        S.partner[rnd * 12 + p] = (unsigned char)q;
        S.partner[rnd * 12 + q] = (unsigned char)p;
    }
    // pass 1: centroid
    double acc[28];
    acc[0] = acc[1] = acc[2] = 0;
    for (int k = tid; k < M; k += EPNP_T) {
        const float* o = obj + 3 * inl[k];
        acc[0] += (double)o[0]; acc[1] += (double)o[1]; acc[2] += (double)o[2];
    }
    block_reduce_sum<3>(acc, S.red, S.out);
    const double c0[3] = {S.out[0] / n, S.out[1] / n, S.out[2] / n};
    __syncthreads();
    // pass 2: PW0^T PW0
    for (int k = 0; k < 6; ++k) acc[k] = 0;
    for (int k = tid; k < M; k += EPNP_T) {
        const float* o = obj + 3 * inl[k];
        const double x = (double)o[0] - c0[0], y = (double)o[1] - c0[1], z = (double)o[2] - c0[2];
        acc[0] += x * x; acc[1] += x * y; acc[2] += x * z; acc[3] += y * y; acc[4] += y * z; acc[5] += z * z;
    }
    block_reduce_sum<6>(acc, S.red, S.out);
    if (tid == 0) {
        const double Sm[9] = {S.out[0], S.out[1], S.out[2], S.out[1], S.out[3], S.out[4], S.out[2], S.out[4], S.out[5]};
        double W[3], U[9], Vt[9], At[9];
        jacobi_svd<3>(Sm, W, U, Vt, At);
        for (int k = 0; k < 3; ++k) S.cws[0][k] = c0[k];
        for (int i = 1; i < 4; ++i) {
            const double kk = sqrt((W[i - 1] > 0 ? W[i - 1] : 0) / n);
            for (int j = 0; j < 3; ++j) S.cws[i][j] = c0[j] + kk * U[3 * j + (i - 1)];
        }
        double cc[9];
        for (int i = 0; i < 3; ++i) for (int j = 1; j < 4; ++j) cc[3 * i + j - 1] = S.cws[j][i] - S.cws[0][i];
        if (!inv3(cc, S.ci)) for (int k = 0; k < 9; ++k) S.ci[k] = nan("");
    }
    __syncthreads();
    phase_stamp(a, b, 4);   // centroid, covariance, 3x3 SVD + control points done
    // pass 3: barycentric coordinates; M^T M in its 4x4-blocks-of-3x3 structure (40 sums) and the moments (16 sums).
    // The 56 sums are split over the two halves of the CTA (28 accumulators per thread instead of 56: the kernel has
    // to fit two CTAs per SM beside the tracker): threads 0-127 take the block pairs (0,0) (0,1) (0,2) (0,3) (1,1) and
    // the moments of alpha_0, alpha_1; threads 128-255 the pairs (1,2) (1,3) (2,2) (2,3) (3,3) and alpha_2, alpha_3.
    double ci[9];
    for (int k = 0; k < 9; ++k) ci[k] = S.ci[k];
    for (int k = 0; k < 28; ++k) acc[k] = 0;
    const int grp = tid >> 7;
    for (int k = tid & 127; k < M; k += EPNP_T / 2) {
        const int id = inl[k];
        const float* o = obj + 3 * id;
        const double X = o[0], Y = o[1], Z = o[2];
        const double dx = X - c0[0], dy = Y - c0[1], dz = Z - c0[2];
        double al[4];
        for (int j = 0; j < 3; ++j) al[1 + j] = ci[3 * j] * dx + ci[3 * j + 1] * dy + ci[3 * j + 2] * dz;
        al[0] = 1.0 - al[1] - al[2] - al[3];
        // undistortPoints (float64) then back to pixels, as cv2's EPnP front end does
        const double fx = cam_at(cam, 0), fy = cam_at(cam, 1), cx = cam_at(cam, 2), cy = cam_at(cam, 3);
        const double u = (((double)img[2 * id] - cx) * ifx) * fx + cx;
        const double v = (((double)img[2 * id + 1] - cy) * ify) * fy + cy;
        const double du = cx - u, dv = cy - v, dd = du * du + dv * dv;
#define EPNP_PAIR(slot, j, l) { const double aa = al[j] * al[l]; acc[4 * (slot)] += aa; acc[4 * (slot) + 1] += aa * du; \
                                acc[4 * (slot) + 2] += aa * dv; acc[4 * (slot) + 3] += aa * dd; }
#define EPNP_MOM(slot, j) { acc[20 + 3 * (slot)] += al[j] * X; acc[20 + 3 * (slot) + 1] += al[j] * Y; acc[20 + 3 * (slot) + 2] += al[j] * Z; \
                            acc[26 + (slot)] += al[j]; }
        if (grp == 0) {
            EPNP_PAIR(0, 0, 0) EPNP_PAIR(1, 0, 1) EPNP_PAIR(2, 0, 2) EPNP_PAIR(3, 0, 3) EPNP_PAIR(4, 1, 1)
            EPNP_MOM(0, 0) EPNP_MOM(1, 1)
            if (k == 0) for (int j = 0; j < 4; ++j) S.alpha0[j] = al[j];
        } else {
            EPNP_PAIR(0, 1, 2) EPNP_PAIR(1, 1, 3) EPNP_PAIR(2, 2, 2) EPNP_PAIR(3, 2, 3) EPNP_PAIR(4, 3, 3)
            EPNP_MOM(0, 2) EPNP_MOM(1, 3)
        }
#undef EPNP_PAIR
#undef EPNP_MOM
    }
    {   // reduce: warps 0-3 hold the first 28 sums, warps 4-7 the other 28
        const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
        for (int k = 0; k < 28; ++k) {
            double x = acc[k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if (lane == 0) S.red[warp * 28 + k] = x;
        }
        __syncthreads();
        if (tid < 56) {
            const int g = tid / 28, kk = tid - 28 * g;
            double x = 0;
            for (int w = 0; w < 4; ++w) x += S.red[(4 * g + w) * 28 + kk];
            // S.out: [0,40) the ten (j <= l) block sums x 4, [40,52) sum alpha_j X, [52,56) sum alpha_j
            const int dst = kk < 20 ? 20 * g + kk : (kk < 26 ? 40 + 6 * g + (kk - 20) : 52 + 2 * g + (kk - 26));
            S.out[dst] = x;
        }
        __syncthreads();
    }
    if (tid < 144) {
        // assemble the 12x12 M^T M, one element per thread: block (jb, lb) of the 4x4 block structure, entry (r, c)
        const int row = tid / 12, col = tid - 12 * row;
        int jb = row / 3, r = row - 3 * jb, lb = col / 3, c = col - 3 * lb;
        if (jb > lb) { int t = jb; jb = lb; lb = t; t = r; r = c; c = t; }      // symmetric: blk(l,j) = blk(j,l)^T
        const int q = jb * 4 - jb * (jb - 1) / 2 + (lb - jb);                    // index of (jb <= lb) in the upper triangle
        const double A = S.out[4 * q], B = S.out[4 * q + 1], Cc = S.out[4 * q + 2], D = S.out[4 * q + 3];
        double v;
        if (r == 0 && c == 0) v = cam_at(cam, 0) * cam_at(cam, 0) * A;
        else if (r == 1 && c == 1) v = cam_at(cam, 1) * cam_at(cam, 1) * A;
        else if (r == 2 && c == 2) v = D;
        else if ((r == 0 && c == 2) || (r == 2 && c == 0)) v = cam_at(cam, 0) * B;
        else if ((r == 1 && c == 2) || (r == 2 && c == 1)) v = cam_at(cam, 1) * Cc;
        else v = 0.0;
        S.jac[0][tid] = v;
    }
    if (tid >= 160 && tid < 172) S.mom_aX[tid - 160] = S.out[40 + tid - 160];
    if (tid >= 172 && tid < 176) S.mom_a[tid - 172] = S.out[52 + tid - 172];
    __syncthreads();
    const double Xbar[3] = {c0[0], c0[1], c0[2]};
    phase_stamp(a, b, 5);   // M^T M assembled
    if (tid < EPNP_JT) {
        const int cur = block_jacobi_eig12(S, tid);
        const double* A = S.jac[cur];
        if (tid < 12) {
            // rank of eigenvalue tid in DESCENDING order (stable); cvSVD(MtM, D, Ut) rows 11, 10, 9, 8 = the four smallest
            const double lam = A[tid * 13];
            int rank = 0;
            for (int m = 0; m < 12; ++m) {
                const double lm = A[m * 13];
                rank += (lm > lam || (lm == lam && m < tid)) ? 1 : 0;
            }
            if (rank >= 8)
                for (int k = 0; k < 12; ++k) S.v4[11 - rank][k] = A[144 + 12 * k + tid];
        }
    }
    __syncthreads();
    phase_stamp(a, b, 6);   // 12x12 eigen-decomposition done
    if (tid < 6) {
        const int pa[6] = {0, 0, 0, 1, 1, 2}, pb[6] = {1, 2, 3, 2, 3, 3};
        const int i = tid;
        double dv[4][3];
        for (int m = 0; m < 4; ++m)
            for (int k = 0; k < 3; ++k) dv[m][k] = S.v4[m][3 * pa[i] + k] - S.v4[m][3 * pb[i] + k];
#define VDOT(p, q) ((p)[0] * (q)[0] + (p)[1] * (q)[1] + (p)[2] * (q)[2])
        double* r = S.L + 10 * i;
        r[0] = VDOT(dv[0], dv[0]); r[1] = 2 * VDOT(dv[0], dv[1]); r[2] = VDOT(dv[1], dv[1]);
        r[3] = 2 * VDOT(dv[0], dv[2]); r[4] = 2 * VDOT(dv[1], dv[2]); r[5] = VDOT(dv[2], dv[2]);
        r[6] = 2 * VDOT(dv[0], dv[3]); r[7] = 2 * VDOT(dv[1], dv[3]); r[8] = 2 * VDOT(dv[2], dv[3]);
        r[9] = VDOT(dv[3], dv[3]);
        const double d[3] = {S.cws[pa[i]][0] - S.cws[pb[i]][0], S.cws[pa[i]][1] - S.cws[pb[i]][1], S.cws[pa[i]][2] - S.cws[pb[i]][2]};
        S.rho[i] = VDOT(d, d);
    }
    __syncthreads();
    // three beta initialisations, one per WARP (their code paths differ: lanes of one warp would run them one
    // after the other), 5 Gauss-Newton steps each, pose from the moments
    if ((tid & 31) == 0 && tid < 96) {
        const int Nn = (tid >> 5) + 1;
        const double* L = S.L;
        double be[4] = {0, 0, 0, 0};
        if (Nn == 1) {
            double A[24], b4[4];
            for (int i = 0; i < 6; ++i) { A[4 * i] = L[10 * i]; A[4 * i + 1] = L[10 * i + 1]; A[4 * i + 2] = L[10 * i + 3]; A[4 * i + 3] = L[10 * i + 6]; }
            qr_lstsq6<4>(A, S.rho, b4);
            if (b4[0] < 0) { be[0] = sqrt(-b4[0]); be[1] = -b4[1] / be[0]; be[2] = -b4[2] / be[0]; be[3] = -b4[3] / be[0]; }
            else { be[0] = sqrt(b4[0]); be[1] = b4[1] / be[0]; be[2] = b4[2] / be[0]; be[3] = b4[3] / be[0]; }
        } else if (Nn == 2) {
            double A[18], b3[3];
            for (int i = 0; i < 6; ++i) { A[3 * i] = L[10 * i]; A[3 * i + 1] = L[10 * i + 1]; A[3 * i + 2] = L[10 * i + 2]; }
            qr_lstsq6<3>(A, S.rho, b3);
            if (b3[0] < 0) { be[0] = sqrt(-b3[0]); be[1] = (b3[2] < 0) ? sqrt(-b3[2]) : 0.0; }
            else { be[0] = sqrt(b3[0]); be[1] = (b3[2] > 0) ? sqrt(b3[2]) : 0.0; }
            if (b3[1] < 0) be[0] = -be[0];
        } else {
            double A[30], b5[5];
            for (int i = 0; i < 6; ++i) for (int k = 0; k < 5; ++k) A[5 * i + k] = L[10 * i + k];
            qr_lstsq6<5>(A, S.rho, b5);
            if (b5[0] < 0) { be[0] = sqrt(-b5[0]); be[1] = (b5[2] < 0) ? sqrt(-b5[2]) : 0.0; }
            else { be[0] = sqrt(b5[0]); be[1] = (b5[2] > 0) ? sqrt(b5[2]) : 0.0; }
            if (b5[1] < 0) be[0] = -be[0];
            be[2] = b5[3] / be[0];
        }
        epnp_gauss_newton(S.L, S.rho, be);
        epnp_pose_from_betas(S, be, n, Xbar, S.Rs[Nn - 1], S.ts[Nn - 1]);
    }
    __syncthreads();
    phase_stamp(a, b, 7);   // betas, Gauss-Newton, three candidate poses done
    // pass 4: mean reprojection error of the three candidates
    acc[0] = acc[1] = acc[2] = 0;
    for (int k = tid; k < M; k += EPNP_T) {
        const int id = inl[k];
        const float* o = obj + 3 * id;
        const double X = o[0], Y = o[1], Z = o[2];
        const double fx = cam_at(cam, 0), fy = cam_at(cam, 1), cx = cam_at(cam, 2), cy = cam_at(cam, 3);
        const double u = (((double)img[2 * id] - cx) * ifx) * fx + cx;
        const double v = (((double)img[2 * id + 1] - cy) * ify) * fy + cy;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const double* R = S.Rs[c];
            const double* t = S.ts[c];
            const double Xc = R[0] * X + R[1] * Y + R[2] * Z + t[0];
            const double Yc = R[3] * X + R[4] * Y + R[5] * Z + t[1];
            const double iZ = 1.0 / (R[6] * X + R[7] * Y + R[8] * Z + t[2]);
            const double ue = cx + fx * Xc * iZ, ve = cy + fy * Yc * iZ;
            const double du = u - ue, dv = v - ve;
            acc[c] += sqrt(du * du + dv * dv);
        }
    }
    block_reduce_sum<3>(acc, S.red, S.out);
    if (tid == 0) {
        const double r1 = S.out[0] / n, r2 = S.out[1] / n, r3 = S.out[2] / n;
        int Nn = 0;
        double rb = r1;
        if (r2 < r1) { Nn = 1; rb = r2; }
        if (r3 < rb) Nn = 2;
        bool fin = true;
        for (int k = 0; k < 9; ++k) fin = fin && isfinite(S.Rs[Nn][k]);
        for (int k = 0; k < 3; ++k) fin = fin && isfinite(S.ts[Nn][k]);
        if (fin) {
            double rv[3];
            R_to_rodrigues(S.Rs[Nn], rv);
            pose_out[0] = rv[0]; pose_out[1] = rv[1]; pose_out[2] = rv[2];
            pose_out[3] = S.ts[Nn][0]; pose_out[4] = S.ts[Nn][1]; pose_out[5] = S.ts[Nn][2];
        }
    }
}

__global__ void __launch_bounds__(EPNP_T)
pnp_epnp_kernel(PnpArgs a)
{
    extern __shared__ __align__(16) uint8_t epnp_smem[];
    EpnpShared& S = *reinterpret_cast<EpnpShared*>(epnp_smem);
    const int b = blockIdx.x;
    if (!a.ok[b]) return;
    const int N = a.n[b];
    const int M = a.n_inliers[b];
    if (N == 4 || M < 4) return;   // N == 4: cv2 returns the direct P3P solve
    epnp_block(a, &a.intr[b].fx, S, a.obj + (size_t)b * a.cap * 3, a.img + (size_t)b * a.cap * 2, a.inliers + (size_t)b * a.cap, M,
               a.pose + (size_t)b * 6, b);
}

// ------------------------------------------------------------------------------------------
// 6. the whole pose chain of one sequence in ONE CTA (the per-frame path: N <= a few thousand correspondences)
// ------------------------------------------------------------------------------------------
// status==1 compaction -> [ 32 cv::RNG subsets -> 32 P3P solves -> score them on every point -> replay cv2's loop ]
// repeated while the adaptive stop still wants hypotheses (typically once: at 10 % outliers cv2 stops after ~5)
// -> winner mask + ordered inlier list -> EPnP refit -> mask over the original landmark slots.
// Same device functions as the multi-kernel path (pnp_solve_one, pnp_is_inlier, epnp_block), so the results are
// the same bits; what disappears is nine dependent launches of one-CTA-per-sequence kernels and the global
// round trips between them (250 us -> one launch), which is what bounds a single sequence and small shards.
#define FUSED_T EPNP_T
#define FUSED_CHUNK 32
#define FUSED_SUB 8       // hypotheses scored between two looks at the adaptive stop
#define FUSED_WIN 256     // raw RNG values looked at per sampling pass

struct PoseFusedShared {
    double h[FUSED_CHUNK * 12];
    double rv[FUSED_CHUNK * 3];
    double win_h[12], win_rv[3];
    int ok[FUSED_CHUNK], cnt[FUSED_CHUNK];
    int smp[FUSED_CHUNK * 4];
    int mod[FUSED_WIN];
    double cam[4];      // the sequence's fx, fy, cx, cy, loaded once per CTA
    int warp_n[8];
    int base, N, niters, max_good, win, it0, pos, nh;
};

// cv::RNG subsets for hypotheses [it0, it0 + nh): one warp; `pos` = position in the raw stream (carried between chunks)
__device__ inline void fused_draw_samples(const PnpArgs& a, PoseFusedShared& F, int b, int N, int nh, int lane)
{
    int i0 = 0;
    int pos = F.pos;
    while (i0 < nh) {
        // residues of the next FUSED_WIN raw values
        for (int k = lane; k < FUSED_WIN; k += 32) F.mod[k] = pos + k < a.n_raw ? (int)(a.rng_raw[pos + k] % (uint32_t)N) : -1;
        __syncwarp();
        const int i = i0 + lane, p = 4 * lane;
        const bool live = i < nh;
        int sv[4] = {0, 0, 0, 0};
        bool bad = false;
        if (live) {
#pragma unroll
            for (int j = 0; j < 4; ++j) sv[j] = F.mod[p + j];
            bad = sv[3] < 0 || sv[0] < 0 || sv[1] < 0 || sv[2] < 0;   // raw table exhausted
#pragma unroll
            for (int j = 1; j < 4; ++j)
#pragma unroll
                for (int m = 0; m < j; ++m) bad = bad || (sv[j] == sv[m]);
        }
        const unsigned stop = __ballot_sync(0xffffffffu, live && bad);
        const int first = stop ? __ffs(stop) - 1 : 32;
        if (live && lane < first) {
#pragma unroll
            for (int j = 0; j < 4; ++j) F.smp[4 * i + j] = sv[j];
        }
        if (first == 32) { pos += 4 * (nh - i0); i0 = nh; break; }
        int npos = 0;
        if (lane == first) {   // getSubset's redraw loop, sequentially, for this one sample (straight from the raw table)
            int q = pos + p, idx[4] = {-1, -1, -1, -1};
            bool okk = true;
            for (int j = 0; j < 4 && okk; ++j) {
                for (;;) {
                    if (q >= a.n_raw) { okk = false; break; }
                    const int v = (int)(a.rng_raw[q++] % (uint32_t)N);
                    bool d = false;
                    for (int m = 0; m < j; ++m) d = d || (idx[m] == v);
                    if (!d) { idx[j] = v; break; }
                }
            }
            if (!okk) {
                idx[0] = idx[1] = idx[2] = idx[3] = -1;
                a.flags[b] |= 1;
                q = a.n_raw;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) F.smp[4 * i + j] = idx[j];
            npos = q;
        }
        pos = __shfl_sync(0xffffffffu, npos, first);
        i0 += first + 1;
        __syncwarp();
    }
    if (lane == 0) F.pos = pos;
}

template <int MIN_CTAS>   // 1: every register the SM has (lowest latency); 2: two CTAs per SM, i.e. room for four tracker CTAs beside one
__global__ void __launch_bounds__(FUSED_T, MIN_CTAS)
pnp_fused_kernel(PnpArgs a, PoseBatchIO io)
{
    extern __shared__ __align__(16) uint8_t fused_smem[];
    PoseFusedShared& F = *reinterpret_cast<PoseFusedShared*>(fused_smem);
    EpnpShared& S = *reinterpret_cast<EpnpShared*>(fused_smem + ((sizeof(PoseFusedShared) + 15) / 16) * 16);
    const int b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* obj = const_cast<float*>(a.obj) + (size_t)b * a.cap * 3;
    float* img = const_cast<float*>(a.img) + (size_t)b * a.cap * 2;
    uint8_t* mask = a.mask + (size_t)b * a.cap;
    int* inl = a.inliers + (size_t)b * a.cap;
    int* orig = io.c_orig ? io.c_orig + (size_t)b * a.cap : nullptr;

    phase_stamp(a, b, 0);
    // ---- 1. status == 1 landmarks, in order (what `matched_pts[tracked]` does in the reference, :282-284) ----
    // (written out rather than cta_compact: this kernel's register allocation is at its limit, <2> spills)
    if (tid == 0) F.base = 0;
    const double cam_r = tid < 4 ? (&a.intr[b].fx)[tid] : 0.0;   // issued now, stored after the compaction (hides the latency)
    __syncthreads();
    if (io.lm_status) {
        const int n = min(max(io.n_lm[b], 0), a.cap);   // a count beyond the slot capacity must not reach the neighbour's arrays
        for (int base = 0; base < n; base += FUSED_T) {
            const int i = base + tid;
            const size_t gi = (size_t)b * a.cap + i;
            const bool keep = i < n && io.lm_status[gi] == 1;
            const unsigned bm = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) F.warp_n[warp] = __popc(bm);
            __syncthreads();
            int off = F.base;
            for (int w = 0; w < warp; ++w) off += F.warp_n[w];
            if (keep) {
                const int o = off + __popc(bm & ((1u << lane) - 1));
                obj[3 * o] = io.lm_obj[3 * gi]; obj[3 * o + 1] = io.lm_obj[3 * gi + 1]; obj[3 * o + 2] = io.lm_obj[3 * gi + 2];
                img[2 * o] = io.lm_next[2 * gi]; img[2 * o + 1] = io.lm_next[2 * gi + 1];
                orig[o] = i;
            }
            __syncthreads();
            if (tid == 0) {
                int tot = 0;
                for (int w = 0; w < FUSED_T / 32; ++w) tot += F.warp_n[w];
                F.base += tot;
            }
            __syncthreads();
        }
        if (tid == 0) const_cast<int*>(a.n)[b] = F.base;
    }
    const int N = io.lm_status ? F.base : min(max(a.n[b], 0), a.cap);
    if (tid == 0) {
        F.niters = N == 4 ? 1 : (N > 4 ? (a.iters > 1 ? a.iters : 1) : 0);
        F.max_good = 0; F.win = -1; F.it0 = 0; F.pos = 0;
    }
    if (tid < 4) F.cam[tid] = cam_r;
    __syncthreads();

    phase_stamp(a, b, 1);   // compaction done
    // ---- 2. RANSAC in chunks of 32 hypotheses; thread 0 replays cv2's loop after each chunk ----
    while (F.it0 < F.niters) {                       // block-uniform: both change only between barriers
        const int it0 = F.it0;
        const int nh = min(FUSED_CHUNK, F.niters - it0);
        if (warp == 0) {
            if (N == 4) { if (lane < 4) F.smp[lane] = lane; }   // count == modelPoints: one direct solve on all points
            else fused_draw_samples(a, F, b, N, nh, lane);
        }
        if (tid < FUSED_CHUNK) F.cnt[tid] = 0;
        __syncthreads();
        phase_stamp(a, b, 9);    // (last chunk) subsets drawn
        // one hypothesis per thread, spread over the warps (P3P branches diverge: 4 per warp, 8 warps issue in parallel)
        if ((tid & 7) == 0) {
            const int h = tid >> 3;
            int okh = 0;
            if (h < nh && F.smp[4 * h] >= 0) okh = pnp_solve_one(F.cam, obj, img, F.smp + 4 * h, F.h + 12 * h, F.rv + 3 * h);
            F.ok[h] = okh;
        }
        __syncthreads();
        phase_stamp(a, b, 10);   // (last chunk) minimal solves done
        // Score eight hypotheses at a time and let thread 0 replay cv2's loop after each eight: cv2 itself stops after
        // ~5 iterations at 10 % outliers, so the usual frame scores 8 hypotheses instead of 32 (the 32 minimal solves run
        // in parallel and cost the latency of one; scoring is what an SM with eight warps is slow at: 31 us for 32).
        for (int h_lo = 0; h_lo < nh; h_lo += FUSED_SUB) {
            const int h_hi = min(h_lo + FUSED_SUB, nh);
            if (N > 4) {
                const double fx = F.cam[0], fy = F.cam[1], cx = F.cam[2], cy = F.cam[3];   // registers for the scoring loop only
                for (int base = 0; base < N; base += FUSED_T) {
                    const int i = base + tid;
                    const bool live = i < N;
                    double X = 0, Y = 0, Z = 0;
                    float iu = 0, iv = 0;
                    if (live) { X = obj[3 * i]; Y = obj[3 * i + 1]; Z = obj[3 * i + 2]; iu = img[2 * i]; iv = img[2 * i + 1]; }
                    // (a float32 pre-test with an error band was tried here: 33 us against 31 us for this exact form on 1000
                    // points x 32 hypotheses -- with eight warps on the SM the phase is bound by issue latency, not by the FP64 pipe)
                    for (int h = h_lo; h < h_hi; ++h) {
                        if (!F.ok[h]) continue;   // block-uniform
                        const bool in = live && pnp_is_inlier(F.h + h * 12, fx, fy, cx, cy, X, Y, Z, iu, iv, a.thr_sq);
                        const unsigned m = __ballot_sync(0xffffffffu, in);
                        if (lane == 0 && m) atomicAdd(&F.cnt[h], __popc(m));
                    }
                }
                __syncthreads();
            }
            if (tid == 0) {
                int niters = F.niters, max_good = F.max_good, win = F.win;
                if (N == 4) { win = F.ok[0] ? 0 : -1; if (win == 0) { for (int k = 0; k < 12; ++k) F.win_h[k] = F.h[k]; for (int k = 0; k < 3; ++k) F.win_rv[k] = F.rv[k]; } }
                else {
                    for (int h = h_lo; h < h_hi && it0 + h < niters; ++h) {
                        if (!F.ok[h]) continue;
                        const int good = F.cnt[h];
                        if (good > (max_good > 3 ? max_good : 3)) {
                            win = it0 + h; max_good = good;
                            niters = ransac_update_num_iters(a.conf, (double)(N - good) / N, 4, niters);
                            for (int k = 0; k < 12; ++k) F.win_h[k] = F.h[12 * h + k];
                            for (int k = 0; k < 3; ++k) F.win_rv[k] = F.rv[3 * h + k];
                        }
                    }
                }
                F.niters = niters; F.max_good = max_good; F.win = win;
                if (h_hi == nh || it0 + h_hi >= niters) F.it0 = it0 + nh;     // this chunk is finished (or the loop is)
            }
            __syncthreads();
            if (it0 + h_hi >= F.niters) break;       // block-uniform: the replay can no longer reach the rest of the chunk
        }
        phase_stamp(a, b, 11);   // (last chunk) scoring + replay done
    }

    phase_stamp(a, b, 2);   // RANSAC chunks done
    // ---- 3. winner mask + ordered inlier list ----
    const int win = F.win;
    int M = 0;
    if (tid == 0) { a.winner[b] = win; a.iters_run[b] = F.niters; F.base = 0; }
    __syncthreads();
    if (win < 0) {
        for (int i = tid; i < a.cap; i += FUSED_T) mask[i] = 0;
        if (tid == 0) { a.n_inliers[b] = 0; a.ok[b] = 0; }
    } else {
        // written out rather than cta_compact, as in step 1
        for (int base = 0; base < a.cap; base += FUSED_T) {
            const int i = base + tid;
            bool in = false;
            if (i < N) in = N == 4 ? true : pnp_is_inlier(F.win_h, cam_at(F.cam, 0), cam_at(F.cam, 1), cam_at(F.cam, 2), cam_at(F.cam, 3), obj[3 * i], obj[3 * i + 1], obj[3 * i + 2], img[2 * i], img[2 * i + 1], a.thr_sq);
            const unsigned bm = __ballot_sync(0xffffffffu, in);
            if (lane == 0) F.warp_n[warp] = __popc(bm);
            __syncthreads();
            int off = F.base;
            for (int w = 0; w < warp; ++w) off += F.warp_n[w];
            if (in) inl[off + __popc(bm & ((1u << lane) - 1))] = i;
            if (i < a.cap) mask[i] = in ? 1 : 0;
            __syncthreads();
            if (tid == 0) {
                int tot = 0;
                for (int w = 0; w < FUSED_T / 32; ++w) tot += F.warp_n[w];
                F.base += tot;
            }
            __syncthreads();
        }
        M = F.base;
        double* pose = a.pose + (size_t)b * 6;
        if (tid == 0) {
            a.n_inliers[b] = M; a.ok[b] = 1;
            // RANSAC model (what cv2 falls back to / returns for N == 4)
            pose[0] = F.win_rv[0]; pose[1] = F.win_rv[1]; pose[2] = F.win_rv[2];
            pose[3] = F.win_h[9]; pose[4] = F.win_h[10]; pose[5] = F.win_h[11];
        }
        __syncthreads();
        phase_stamp(a, b, 3);   // winner mask + inlier list done
        // ---- 4. EPnP refit on the inliers (N == 4: cv2 returns the direct P3P solve) ----
        if (N != 4 && M >= 4) epnp_block(a, F.cam, S, obj, img, inl, M, pose, b);
    }
    phase_stamp(a, b, 8);   // EPnP done
    // ---- 5. inlier mask over the ORIGINAL landmark slots (:346) ----
    if (io.mask_out) {
        __syncthreads();
        uint8_t* mo = io.mask_out + (size_t)b * a.cap;
        for (int i = tid; i < a.cap; i += FUSED_T) mo[i] = 0;
        __syncthreads();
        for (int k = tid; k < M; k += FUSED_T) mo[orig[inl[k]]] = 1;
        if (tid == 0) { io.n_inl_out[b] = M; io.ok_out[b] = win >= 0 ? 1 : 0; }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
void vo_rng_raw_stream(uint32_t* out, int n)
{
    // cv::RNG((uint64)-1): state = (uint32)state * 4164903690 + (state >> 32)
    uint64_t st = 0xFFFFFFFFFFFFFFFFull;
    for (int i = 0; i < n; ++i) {
        st = (uint64_t)(uint32_t)st * 4164903690u + (st >> 32);
        out[i] = (uint32_t)st;
    }
}

int vo_rng_table(b200vo_ctx* ctx, int n, const uint32_t** d_table)
{
    if (n > ctx->n_rng) {
        const int cap = n + n / 2 + 1024;
        uint32_t* h = (uint32_t*)malloc((size_t)cap * sizeof(uint32_t));
        if (!h) return vo_set_err(ctx, B200VO_E_NOMEM, "host alloc");
        vo_rng_raw_stream(h, cap);
        int rc = vo_reserve(ctx, ctx->d_rng, (size_t)cap * sizeof(uint32_t));
        if (rc == 0) {
            cudaError_t e = cudaMemcpyAsync(ctx->d_rng.p, h, (size_t)cap * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) rc = vo_cuda_fail(ctx, e, "rng table upload");
        }
        free(h);
        if (rc) return rc;
        ctx->n_rng = cap;
    }
    *d_table = (const uint32_t*)ctx->d_rng.p;
    return 0;
}

size_t vo_pnp_workspace_bytes(int batch, int cap, int iters)
{
    size_t b = 0;
    b += vo_align((size_t)batch * iters * 4 * sizeof(int), 256);       // samples
    b += vo_align((size_t)batch * iters * 12 * sizeof(double), 256);   // hyp
    b += vo_align((size_t)batch * iters * 3 * sizeof(double), 256);    // hyp_rvec
    b += 2 * vo_align((size_t)batch * iters * sizeof(int), 256);       // hyp_ok, counts
    b += 4 * vo_align((size_t)batch * sizeof(int), 256);               // winner, iters_run, n_inliers, ok_ws
    b += vo_align((size_t)batch * 3 * sizeof(int), 256);               // flags | ticket | need
    return b;
}

void vo_pnp_carve_workspace(PnpArgs& a, void* ws)
{
    uint8_t* p = (uint8_t*)ws;
    auto take = [&](size_t bytes) { void* r = p; p += vo_align(bytes, 256); return r; };
    a.samples = (int*)take((size_t)a.batch * a.iters * 4 * sizeof(int));
    a.hyp = (double*)take((size_t)a.batch * a.iters * 12 * sizeof(double));
    a.hyp_rvec = (double*)take((size_t)a.batch * a.iters * 3 * sizeof(double));
    a.hyp_ok = (int*)take((size_t)a.batch * a.iters * sizeof(int));
    a.counts = (int*)take((size_t)a.batch * a.iters * sizeof(int));
    a.winner = (int*)take((size_t)a.batch * sizeof(int));
    a.iters_run = (int*)take((size_t)a.batch * sizeof(int));
    a.n_inliers = (int*)take((size_t)a.batch * sizeof(int));
    a.flags = (int*)take((size_t)a.batch * 3 * sizeof(int));
    a.ticket = a.flags + a.batch;
    a.need = a.flags + 2 * a.batch;
    a.ok_ws = (uint8_t*)take((size_t)a.batch * sizeof(int));
}

bool vo_pnp_fused_ok(const PnpArgs& a, bool gen_samples)
{
    return gen_samples && !a.full_counts && a.cap <= VO_PNP_FUSED_MAX_N;
}

int vo_pnp_fused_launch(b200vo_ctx* ctx, const PnpArgs& a, const PoseBatchIO& io, cudaStream_t stream)
{
    if (a.batch <= 0) return 0;
    const size_t smem = ((sizeof(PoseFusedShared) + 15) / 16) * 16 + sizeof(EpnpShared);
    static_assert(((sizeof(PoseFusedShared) + 15) / 16) * 16 + sizeof(EpnpShared) <= 48 * 1024, "static limit of dynamic shared memory");
    // few sequences: the chain's latency is the step (single sequence, small shards) -> the unconstrained build;
    // many: it runs beside the candidate tracker and must leave it registers -> two CTAs per SM
    const bool wide = 2 * a.batch <= ctx->num_sms;
    VO_CUDA(ctx, cudaMemsetAsync(a.flags, 0, (size_t)a.batch * 3 * sizeof(int), stream));
    if (wide) pnp_fused_kernel<1><<<a.batch, FUSED_T, smem, stream>>>(a, io);
    else pnp_fused_kernel<2><<<a.batch, FUSED_T, smem, stream>>>(a, io);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

int vo_pnp_launch(b200vo_ctx* ctx, const PnpArgs& a, bool gen_samples, cudaStream_t stream)
{
    if (a.batch <= 0) return 0;
    if (vo_pnp_fused_ok(a, gen_samples)) return vo_pnp_fused_launch(ctx, a, PoseBatchIO{}, stream);
    VO_CUDA(ctx, cudaMemsetAsync(a.flags, 0, (size_t)a.batch * 3 * sizeof(int), stream));
    if (gen_samples) {
        const size_t smem = (size_t)a.n_raw * sizeof(int);
        if (smem > 48 * 1024)
            VO_CUDA(ctx, cudaFuncSetAttribute(ransac_samples_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ransac_samples_kernel<4><<<a.batch, 128, smem, stream>>>(a.rng_raw, a.n_raw, a.n, a.iters, a.samples, a.flags);
        ctx->launches++;
    }
    // head chunk: the first PNP_HEAD hypotheses; its last scoring CTA per sequence leaves need[b].
    // tail chunk: whatever the replay can still reach (CTAs beyond need[b] exit at once).
    const int head_n = (a.full_counts || a.iters < PNP_HEAD) ? a.iters : PNP_HEAD;
    for (int part = 0; part < 2; ++part) {
        PnpArgs c = a;
        c.head = part == 0;
        c.h_begin = part == 0 ? 0 : head_n;
        c.h_end = part == 0 ? head_n : a.iters;
        const int nh = c.h_end - c.h_begin;
        if (nh <= 0) continue;
        dim3 g1((nh + 63) / 64, a.batch);
        pnp_solve_kernel<<<g1, 64, 0, stream>>>(c);
        dim3 g2((a.cap + 255) / 256, (nh + SCORE_HT - 1) / SCORE_HT, a.batch);
        pnp_score_kernel<<<g2, 256, 0, stream>>>(c);
        ctx->launches += 2;
    }
    pnp_select_kernel<<<a.batch, 256, 0, stream>>>(a);
    ctx->launches++;
    {
        const size_t smem = sizeof(EpnpShared);
        pnp_epnp_kernel<<<a.batch, EPNP_T, smem, stream>>>(a);
        ctx->launches++;
    }
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}
