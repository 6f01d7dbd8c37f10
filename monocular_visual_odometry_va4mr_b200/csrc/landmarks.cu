// The two components next to the hot path (SURVEY.md 8f), downstream of the tracker and of
// goodFeaturesToTrack in the reference's per-frame loop:
//   f2  candidate min-distance filter, reference VisualOdometryPipeLine.py:258
//         valid[i] = np.all(np.linalg.norm(pts[i,:] - self.potential_keys, axis=1) > min_dist)
//       (float32: squares, sum and square root rounded as numpy rounds them);
//   f1  triangulate_landmarks, reference :107-206: age gate (:171-174), bearing-angle gate
//       (:117-147), cv2.triangulatePoints (:188-193: 4x4 DLT, OpenCV's small-matrix Jacobi SVD,
//       float32 homogeneous output), de-homogenisation (:194), depth window in both cameras
//       (:149-168); accepted landmarks and their keypoints appended in candidate order.
// The reference spends ~67 ms (f1) and ~48 ms (f2) per frame on these in Python loops
// (SURVEY.md 8f); here each is one or two small launches.
#include "landmarks.cuh"
#include "mathdev.cuh"

using namespace vo;

__device__ __forceinline__ void invert_pose(const double* cw, double* R, double* t)
{
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) R[3 * i + j] = cw[3 * j + i];
#pragma unroll
    for (int i = 0; i < 3; ++i) t[i] = -(R[3 * i] * cw[9] + R[3 * i + 1] * cw[10] + R[3 * i + 2] * cw[11]);
}
__device__ __forceinline__ void proj_matrix(const double* K, const double* R, const double* t, double* P)
{
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) P[4 * i + j] = K[3 * i] * R[j] + K[3 * i + 1] * R[3 + j] + K[3 * i + 2] * R[6 + j];
        P[4 * i + 3] = K[3 * i] * t[0] + K[3 * i + 1] * t[1] + K[3 * i + 2] * t[2];
    }
}

// ---- f1: one thread per candidate ----
__device__ __forceinline__ void triangulate_one(const TriArgs& a, int i)
{
    a.keep[i] = 1;
    const int fp = a.first_pose[i];
    if (a.n_poses > 1 && a.n_poses - fp <= a.min_frames) return;
    if (fp < 0 || fp >= a.n_poses) { atomicOr(a.flags, 1); return; }
    double past[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) past[k] = a.poses[12 * fp + k];
    const double u = a.keys[2 * i], v = a.keys[2 * i + 1], u0 = a.first_keys[2 * i], v0 = a.first_keys[2 * i + 1];
    {   // bearing angle between the two viewing rays (check_baseline)
        const double ax = a.Ki[0] * u + a.Ki[2], ay = a.Ki[4] * v + a.Ki[5], az = 1.0;
        double rel[9], M[9];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) rel[3 * r + c] = past[r] * a.cur[c] + past[3 + r] * a.cur[3 + c] + past[6 + r] * a.cur[6 + c];
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
            for (int c = 0; c < 3; ++c) M[3 * r + c] = rel[3 * r] * a.Ki[c] + rel[3 * r + 1] * a.Ki[3 + c] + rel[3 * r + 2] * a.Ki[6 + c];
        const double bx = M[0] * u0 + M[1] * v0 + M[2], by = M[3] * u0 + M[4] * v0 + M[5], bz = M[6] * u0 + M[7] * v0 + M[8];
        double cs = (ax * bx + ay * by + az * bz) / (sqrt(ax * ax + ay * ay + az * az) * sqrt(bx * bx + by * by + bz * bz));
        cs = cs < -1.0 ? -1.0 : (cs > 1.0 ? 1.0 : cs);
        const double alpha = acos(cs) * (180.0 / 3.14159265358979323846);
        if (alpha < a.min_angle_deg) return;
    }
    double Rc[9], tc[3], Pc[12], Rp[9], tp[3], Pp[12];
    invert_pose(a.cur, Rc, tc);
    proj_matrix(a.K, Rc, tc, Pc);
    invert_pose(past, Rp, tp);
    proj_matrix(a.K, Rp, tp, Pp);
    double A[16], W[4], U[16], Vt[16], At[16];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        A[k] = u0 * Pp[8 + k] - Pp[k];
        A[4 + k] = v0 * Pp[8 + k] - Pp[4 + k];
        A[8 + k] = u * Pc[8 + k] - Pc[k];
        A[12 + k] = v * Pc[8 + k] - Pc[4 + k];
    }
    jacobi_svd<4>(A, W, U, Vt, At);
    const float X0 = (float)Vt[12], X1 = (float)Vt[13], X2 = (float)Vt[14], X3 = (float)Vt[15];
    const float L0 = __fdiv_rn(X0, X3), L1 = __fdiv_rn(X1, X3), L2 = __fdiv_rn(X2, X3);
    const double zc = Rc[6] * (double)L0 + Rc[7] * (double)L1 + Rc[8] * (double)L2 + tc[2];
    const double zp = Rp[6] * (double)L0 + Rp[7] * (double)L1 + Rp[8] * (double)L2 + tp[2];
    if (zc > a.min_dist && zp > a.min_dist && zc < a.max_dist && zp < a.max_dist) {
        a.keep[i] = 0;
        a.lm_slot[3 * i] = L0; a.lm_slot[3 * i + 1] = L1; a.lm_slot[3 * i + 2] = L2;
    }
}

// ---- f1 and f2 for a batch of sequences (SURVEY 8f "batched f1/f2 on the resident batch state") in one launch each;
// blockIdx.y = sequence, ragged counts per sequence.  The per-sequence entry points are the batch of one ----
__device__ __forceinline__ TriArgs tri_sequence(const TriBatchArgs& b, int s)
{
    TriArgs a = b.common;
    a.K = b.intr[s].K; a.Ki = b.intr[s].Ki;
    const size_t o = (size_t)s * b.cap;
    a.n = min(max(b.n[s], 0), b.cap);
    a.n_poses = min(max(b.n_poses[s], 0), b.pose_cap);
    for (int k = 0; k < 12; ++k) a.cur[k] = b.cur[12 * s + k];
    a.first_keys = b.first_keys + 2 * o; a.keys = b.keys + 2 * o; a.first_pose = b.first_pose + o;
    a.poses = b.poses + (size_t)s * b.pose_cap * 12;
    a.keep = b.keep + o; a.lm_slot = b.lm_slot + 3 * o; a.out_lm = b.out_lm + 3 * o; a.out_kp = b.out_kp + 2 * o;
    a.n_new = b.n_new + s; a.flags = b.flags + s;
    return a;
}

__global__ void __launch_bounds__(64)
triangulate_batch_kernel(TriBatchArgs b)
{
    const TriArgs a = tri_sequence(b, blockIdx.y);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (a.n_poses < 1) { if (i < a.n) a.keep[i] = 1; return; }
    if (i < a.n) triangulate_one(a, i);
}

// ordered compaction of the accepted candidates (keep == 0): one CTA per sequence
__global__ void __launch_bounds__(1024)
triangulate_compact_batch_kernel(TriBatchArgs b)
{
    const TriArgs a = tri_sequence(b, blockIdx.x);
    const int cnt = cta_compact<1024>(a.n, [&](int i) { return a.keep[i] == 0; }, [&](int i, int o) {
        a.out_lm[3 * o] = a.lm_slot[3 * i]; a.out_lm[3 * o + 1] = a.lm_slot[3 * i + 1]; a.out_lm[3 * o + 2] = a.lm_slot[3 * i + 2];
        a.out_kp[2 * o] = a.keys[2 * i]; a.out_kp[2 * o + 1] = a.keys[2 * i + 1];
    });
    if (threadIdx.x == 0) *a.n_new = cnt;
}

// f2: one warp per new corner, lanes stride over the existing candidates
__global__ void __launch_bounds__(256)
min_distance_batch_kernel(const float2* __restrict__ pts, const int* __restrict__ n, int n_cap, const float2* __restrict__ existing,
                          const int* __restrict__ m, int m_cap, float min_dist, uint8_t* __restrict__ valid)
{
    const int s = blockIdx.y;
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= min(max(n[s], 0), n_cap)) return;
    const float2 p = pts[(size_t)s * n_cap + i];
    const float2* ex = existing + (size_t)s * m_cap;
    const int ms = min(max(m[s], 0), m_cap);
    bool ok = true;
    for (int j0 = 0; j0 < ms; j0 += 32) {
        const int j = j0 + lane;
        if (j < ms) {
            const float2 q = ex[j];
            const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y);
            const float d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
            ok = d > min_dist;           // NaN compares false, as in numpy
        }
        if (!__all_sync(0xffffffffu, ok)) { ok = false; break; }
    }
    if (lane == 0) valid[(size_t)s * n_cap + i] = ok ? 1 : 0;
}

void vo_tri_common(TriArgs& c, double min_dist, double max_dist, double min_angle_deg, int min_frames)
{
    c.min_dist = min_dist; c.max_dist = max_dist; c.min_angle_deg = min_angle_deg;
    c.min_frames = min_frames;
}

int vo_triangulate_batch_launch(b200vo_ctx* ctx, const TriBatchArgs& b, int batch, cudaStream_t stream)
{
    triangulate_batch_kernel<<<dim3((b.cap + 63) / 64, batch), 64, 0, stream>>>(b);
    triangulate_compact_batch_kernel<<<batch, 1024, 0, stream>>>(b);
    ctx->launches += 2;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

int vo_min_distance_batch_launch(b200vo_ctx* ctx, int batch, const float* pts, const int* n, int n_cap, const float* existing,
                                 const int* m, int m_cap, float min_dist, uint8_t* valid, cudaStream_t stream)
{
    min_distance_batch_kernel<<<dim3((n_cap * 32 + 255) / 256, batch), 256, 0, stream>>>(
        (const float2*)pts, n, n_cap, (const float2*)existing, m, m_cap, min_dist, valid);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// Body of both f2 entry points: stages pts (batch, n_cap, 2), existing (batch, m_cap, 2) and the counts in the pinned
// block, runs the kernel and waits.  *valid_h points at the result in the pinned block: uint8 (batch, n_cap), rows >= n[s] 0.
static int min_distance_staged(b200vo_ctx* ctx, int batch, const float* pts, const int32_t* n, int n_cap, const float* existing,
                               const int32_t* m, int m_cap, float min_dist, const uint8_t** valid_h)
{
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const int mc = m_cap > 0 ? m_cap : 1;
    const size_t b_p = vo_align((size_t)batch * n_cap * 8, 256), b_e = vo_align((size_t)batch * mc * 8, 256);
    const size_t b_c = vo_align((size_t)batch * 4, 256), b_v = vo_align((size_t)batch * n_cap, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[6], b_p + b_e + 2 * b_c + b_v));
    VO_TRY(vo_reserve_pinned(ctx, b_p + b_e + 2 * b_c + b_v));
    uint8_t* d = (uint8_t*)ctx->d_scratch[6].p;
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    memcpy(hp, pts, (size_t)batch * n_cap * 8);
    if (m_cap > 0) memcpy(hp + b_p, existing, (size_t)batch * m_cap * 8);
    memcpy(hp + b_p + b_e, n, (size_t)batch * 4);
    memcpy(hp + b_p + b_e + b_c, m, (size_t)batch * 4);
    VO_CUDA(ctx, cudaMemcpyAsync(d, hp, b_p + b_e + 2 * b_c, cudaMemcpyHostToDevice, ctx->stream));
    uint8_t* dv = d + b_p + b_e + 2 * b_c;
    bool full = true;   // every row is live (the batch of one): the kernel writes all of them, nothing to clear
    for (int s = 0; s < batch; ++s) full = full && n[s] >= n_cap;
    if (!full) VO_CUDA(ctx, cudaMemsetAsync(dv, 0, b_v, ctx->stream));
    VO_TRY(vo_min_distance_batch_launch(ctx, batch, (const float*)d, (const int*)(d + b_p + b_e), n_cap, (const float*)(d + b_p),
                                        (const int*)(d + b_p + b_e + b_c), m_cap, min_dist, dv, ctx->stream));
    uint8_t* ho = hp + b_p + b_e + 2 * b_c;
    VO_CUDA(ctx, cudaMemcpyAsync(ho, dv, (size_t)batch * n_cap, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    *valid_h = ho;
    return 0;
}

// The results of triangulate_staged in the pinned block, laid out as the batched entry point returns them
struct TriResults {
    const uint8_t* keep;       // [batch][cap] too_short_baseline
    const float* lm;           // [batch][cap][3] compacted per sequence
    const float* kp;           // [batch][cap][2]
    const int* n_new;          // [batch]
    const int* flags;          // [batch] bit0: first_pose out of range
};

// Body of both f1 entry points: stages the (batch, cap, ...) inputs in the pinned block, runs the two kernels and waits.
static int triangulate_staged(b200vo_ctx* ctx, const double K[9], double min_dist, double max_dist, double min_baseline_angle_deg,
                              int min_baseline_frames, int batch, int cap, const float* first_keys, const float* keys,
                              const int32_t* first_pose, const int32_t* n, const double* poses_cw, const int32_t* n_poses, int pose_cap,
                              const double* cur_pose_cw, TriResults* res)
{
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    TriBatchArgs b{};
    vo_tri_common(b.common, min_dist, max_dist, min_baseline_angle_deg, min_baseline_frames);
    VO_TRY(vo_intrinsics_uniform(ctx, K, VO_BOOT_EMAT_THR, batch, &b.intr));   // one K for every sequence
    b.cap = cap; b.pose_cap = pose_cap;
    const size_t nc = (size_t)batch * cap;
    const size_t b_k = vo_align(nc * 8, 256), b_fp = vo_align(nc * 4, 256), b_ps = vo_align((size_t)batch * pose_cap * 96, 256);
    const size_t b_cnt = vo_align((size_t)batch * 4, 256), b_cur = vo_align((size_t)batch * 96, 256);
    const size_t b_keep = vo_align(nc, 256), b_lm = vo_align(nc * 12, 256);
    const size_t in_bytes = 2 * b_k + b_fp + b_ps + 2 * b_cnt + b_cur, out_bytes = b_keep + b_lm + b_k + 2 * b_cnt;
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[7], in_bytes + out_bytes + b_lm));
    VO_TRY(vo_reserve_pinned(ctx, in_bytes + out_bytes));
    uint8_t* d = (uint8_t*)ctx->d_scratch[7].p;
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    size_t o = 0;
    memcpy(hp + o, first_keys, nc * 8); b.first_keys = (const float*)(d + o); o += b_k;
    memcpy(hp + o, keys, nc * 8); b.keys = (const float*)(d + o); o += b_k;
    memcpy(hp + o, first_pose, nc * 4); b.first_pose = (const int*)(d + o); o += b_fp;
    memcpy(hp + o, poses_cw, (size_t)batch * pose_cap * 96); b.poses = (const double*)(d + o); o += b_ps;
    memcpy(hp + o, n, (size_t)batch * 4); b.n = (const int*)(d + o); o += b_cnt;
    memcpy(hp + o, n_poses, (size_t)batch * 4); b.n_poses = (const int*)(d + o); o += b_cnt;
    memcpy(hp + o, cur_pose_cw, (size_t)batch * 96); b.cur = (const double*)(d + o); o += b_cur;
    VO_CUDA(ctx, cudaMemcpyAsync(d, hp, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    uint8_t* dout = d + in_bytes;
    b.keep = dout; b.out_lm = (float*)(dout + b_keep); b.out_kp = (float*)(dout + b_keep + b_lm);
    b.n_new = (int*)(dout + b_keep + b_lm + b_k); b.flags = (int*)(dout + b_keep + b_lm + b_k + b_cnt);
    b.lm_slot = (float*)(dout + out_bytes);
    VO_CUDA(ctx, cudaMemsetAsync(dout, 0, out_bytes, ctx->stream));
    VO_TRY(vo_triangulate_batch_launch(ctx, b, batch, ctx->stream));
    uint8_t* ho = hp + in_bytes;
    VO_CUDA(ctx, cudaMemcpyAsync(ho, dout, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    res->keep = ho; res->lm = (const float*)(ho + b_keep); res->kp = (const float*)(ho + b_keep + b_lm);
    res->n_new = (const int*)(ho + b_keep + b_lm + b_k); res->flags = (const int*)(ho + b_keep + b_lm + b_k + b_cnt);
    return 0;
}

extern "C" int b200vo_min_distance_mask(b200vo_ctx* ctx, const float* pts, int n, const float* existing, int m,
                                        float min_dist, uint8_t* valid)
{
    if (!ctx || n < 0 || m < 0 || (n > 0 && (!pts || !valid)) || (m > 0 && !existing)) return B200VO_E_BADARG;
    if (n == 0) return 0;
    const uint8_t* h;
    VO_TRY(min_distance_staged(ctx, 1, pts, &n, n, existing, &m, m, min_dist, &h));
    memcpy(valid, h, (size_t)n);
    return 0;
}

extern "C" int b200vo_triangulate_landmarks(b200vo_ctx* ctx, const double K[9], double min_dist, double max_dist,
                                            double min_baseline_angle_deg, int min_baseline_frames,
                                            const float* first_keys, const float* keys, const int32_t* first_pose, int n,
                                            const double* poses_cw, int n_poses, const double cur_pose_cw[12],
                                            uint8_t* too_short_baseline, float* new_landmarks, float* new_keypoints,
                                            int* n_new)
{
    if (!ctx || !K || !cur_pose_cw || !n_new || n < 0 || n_poses < 1 || !poses_cw) return B200VO_E_BADARG;
    *n_new = 0;
    if (n == 0) return 0;
    if (!first_keys || !keys || !first_pose || !too_short_baseline || !new_landmarks || !new_keypoints)
        return vo_set_err(ctx, B200VO_E_BADARG, "null pointer");
    TriResults r;
    VO_TRY(triangulate_staged(ctx, K, min_dist, max_dist, min_baseline_angle_deg, min_baseline_frames, 1, n, first_keys, keys,
                              first_pose, &n, poses_cw, &n_poses, n_poses, cur_pose_cw, &r));
    if (r.flags[0] & 1) return vo_set_err(ctx, B200VO_E_BADARG, "first_pose index outside [0, n_poses)");
    const int cnt = r.n_new[0];
    memcpy(too_short_baseline, r.keep, (size_t)n);
    memcpy(new_landmarks, r.lm, (size_t)cnt * 12);
    memcpy(new_keypoints, r.kp, (size_t)cnt * 8);
    *n_new = cnt;
    return 0;
}

// Batched f2: the candidate min-distance filter (:258) for every sequence of a batch in one launch.
// pts float32 (batch, n_cap, 2) with n[batch] live rows, existing float32 (batch, m_cap, 2) with m[batch]; valid uint8 (batch, n_cap).
extern "C" int b200vo_batch_min_distance_mask(b200vo_ctx* ctx, int batch, const float* pts, const int32_t* n, int n_cap,
                                              const float* existing, const int32_t* m, int m_cap, float min_dist, uint8_t* valid)
{
    if (!ctx || batch < 1 || n_cap < 1 || m_cap < 0 || !pts || !n || !m || !valid || (m_cap > 0 && !existing)) return B200VO_E_BADARG;
    const uint8_t* h;
    VO_TRY(min_distance_staged(ctx, batch, pts, n, n_cap, existing, m, m_cap, min_dist, &h));
    memcpy(valid, h, (size_t)batch * n_cap);
    return 0;
}

// Batched f1: the candidate loop of triangulate_landmarks (:170-204) for every sequence of a batch: two launches.
// Per sequence s: n[s] candidates in rows [0, n[s]) of the (batch, cap, ...) arrays, n_poses[s] stored poses in
// poses_cw (batch, pose_cap, 12), the current pose cur_pose_cw (batch, 12).  Outputs: too_short_baseline uint8 (batch, cap),
// new_landmarks float32 (batch, cap, 3) / new_keypoints float32 (batch, cap, 2) compacted per sequence, n_new int32 (batch).
extern "C" int b200vo_batch_triangulate_landmarks(b200vo_ctx* ctx, const double K[9], double min_dist, double max_dist,
                                                  double min_baseline_angle_deg, int min_baseline_frames, int batch, int cap,
                                                  const float* first_keys, const float* keys, const int32_t* first_pose,
                                                  const int32_t* n, const double* poses_cw, const int32_t* n_poses, int pose_cap,
                                                  const double* cur_pose_cw, uint8_t* too_short_baseline, float* new_landmarks,
                                                  float* new_keypoints, int32_t* n_new)
{
    if (!ctx || !K || batch < 1 || cap < 1 || pose_cap < 1 || !first_keys || !keys || !first_pose || !n || !poses_cw || !n_poses ||
        !cur_pose_cw || !too_short_baseline || !new_landmarks || !new_keypoints || !n_new)
        return B200VO_E_BADARG;
    TriResults r;
    VO_TRY(triangulate_staged(ctx, K, min_dist, max_dist, min_baseline_angle_deg, min_baseline_frames, batch, cap, first_keys, keys,
                              first_pose, n, poses_cw, n_poses, pose_cap, cur_pose_cw, &r));
    for (int s = 0; s < batch; ++s)
        if (r.flags[s] & 1) return vo_set_err(ctx, B200VO_E_BADARG, "sequence %d: first_pose index outside [0, n_poses)", s);
    const size_t nc = (size_t)batch * cap;
    memcpy(too_short_baseline, r.keep, nc);
    memcpy(new_landmarks, r.lm, nc * 12);
    memcpy(new_keypoints, r.kp, nc * 8);
    memcpy(n_new, r.n_new, (size_t)batch * 4);
    return 0;
}

// ------------------------------------------------------------------------------------------
// f3: cv2.recoverPose(E, points1, points2, K) at reference :315 (default distanceThresh = 50), for a batch of independent
// (E, point set) pairs; the sequence is taken from the grid and one call is the batch of one.
//   recover_decompose_kernel   one thread: SVD of E (OpenCV's small-matrix Jacobi), det sign fix,
//                              R1 = U W Vt, R2 = U W^T Vt, t = U[:,2]; the four [R | +-t]
//   recover_cheirality_kernel  one thread per (point, pose): 4x4 DLT with P0 = [I|0] on
//                              K-normalised float64 points, Jacobi SVD, the three sign / depth
//                              tests -> mask 0 / 255; warp-aggregated counts
//   recover_pick_kernel        the winner: most passing points, ties in the order 1, 2, 3, 4
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double det3d(const double* M)
{
    return M[0] * (M[4] * M[8] - M[5] * M[7]) - M[1] * (M[3] * M[8] - M[5] * M[6]) + M[2] * (M[3] * M[7] - M[4] * M[6]);
}
__device__ __forceinline__ void mat3_mul(const double* A, const double* B, double* C)
{
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) C[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
}

__global__ void recover_decompose_kernel(RecArgs a)
{
    const int s = blockIdx.x;
    if (threadIdx.x != 0 || (a.valid && !a.valid[a.valid_stride * s])) return;
    double E[9], W[3], U[9], Vt[9], At[9], T[9], R1[9], R2[9];
    for (int k = 0; k < 9; ++k) E[k] = a.E[9 * s + k];
    jacobi_svd<3>(E, W, U, Vt, At);
    if (det3d(U) < 0) for (int k = 0; k < 9; ++k) U[k] = -U[k];
    if (det3d(Vt) < 0) for (int k = 0; k < 9; ++k) Vt[k] = -Vt[k];
    const double Wm[9] = {0, 1, 0, -1, 0, 0, 0, 0, 1}, Wt[9] = {0, -1, 0, 1, 0, 0, 0, 0, 1};
    mat3_mul(U, Wm, T); mat3_mul(T, Vt, R1);
    mat3_mul(U, Wt, T); mat3_mul(T, Vt, R2);
    const double t[3] = {U[2], U[5], U[8]};
    double* poses = a.poses + 48 * s;
    for (int h = 0; h < 4; ++h) {
        const double* R = (h & 1) ? R2 : R1;
        const double sg = h < 2 ? 1.0 : -1.0;
        for (int k = 0; k < 9; ++k) poses[12 * h + k] = R[k];
        for (int k = 0; k < 3; ++k) poses[12 * h + 9 + k] = sg * t[k];
    }
}

__global__ void __launch_bounds__(128)
recover_cheirality_kernel(RecArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int h = blockIdx.y, s = blockIdx.z;
    const int n = a.n[s];
    if (blockIdx.x * blockDim.x >= n) return;
    const size_t po = (size_t)s * a.cap;
    const double* poses = a.poses + 48 * s;
    bool ok = false;
    if (i < n) {
        double P[12];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int c = 0; c < 3; ++c) P[4 * r + c] = poses[12 * h + 3 * r + c];
            P[4 * r + 3] = poses[12 * h + 9 + r];
        }
        const float* p1 = a.p1 + 2 * po;
        const float* p2 = a.p2 + 2 * po;
        const VoIntrinsics& c = a.intr[s];
        const double x1 = ((double)p1[2 * i] - c.cx) / c.fx, y1 = ((double)p1[2 * i + 1] - c.cy) / c.fy;
        const double x2 = ((double)p2[2 * i] - c.cx) / c.fx, y2 = ((double)p2[2 * i + 1] - c.cy) / c.fy;
        double A[16] = {-1, 0, x1, 0, 0, -1, y1, 0, 0, 0, 0, 0, 0, 0, 0, 0}, W[4], U[16], Vt[16], At[16];
#pragma unroll
        for (int k = 0; k < 4; ++k) { A[8 + k] = x2 * P[8 + k] - P[k]; A[12 + k] = y2 * P[8 + k] - P[4 + k]; }
        jacobi_svd<4>(A, W, U, Vt, At);
        double Q0 = Vt[12], Q1 = Vt[13], Q2 = Vt[14], Q3 = Vt[15];
        ok = Q2 * Q3 > 0;
        Q0 /= Q3; Q1 /= Q3; Q2 /= Q3; Q3 /= Q3;
        ok = ok && (Q2 < a.dist);
        const double z = P[8] * Q0 + P[9] * Q1 + P[10] * Q2 + P[11] * Q3;
        ok = ok && (z > 0) && (z < a.dist);
        if (a.masks) a.masks[4 * po + (size_t)h * a.cap + i] = ok ? 255 : 0;
    }
    const unsigned bm = __ballot_sync(0xffffffffu, ok);
    if ((threadIdx.x & 31) == 0 && bm) atomicAdd(a.good + 4 * s + h, __popc(bm));
}

__global__ void recover_pick_kernel(RecArgs a)
{
    const int s = blockIdx.x;
    if (threadIdx.x != 0) return;
    const int* good = a.good + 4 * s;
    int win;
    if (good[0] >= good[1] && good[0] >= good[2] && good[0] >= good[3]) win = 0;
    else if (good[1] >= good[0] && good[1] >= good[2] && good[1] >= good[3]) win = 1;
    else if (good[2] >= good[0] && good[2] >= good[1] && good[2] >= good[3]) win = 2;
    else win = 3;
    for (int k = 0; k < 12; ++k) a.Rt[12 * s + k] = a.poses[48 * s + 12 * win + k];
    a.win[2 * s] = win; a.win[2 * s + 1] = good[win];
}

int vo_recover_pose_batch_launch(b200vo_ctx* ctx, const RecArgs& a, int nseq, int max_n, cudaStream_t stream)
{
    VO_CUDA(ctx, cudaMemsetAsync(a.good, 0, (size_t)nseq * 16, stream));
    recover_decompose_kernel<<<nseq, 32, 0, stream>>>(a);
    if (max_n > 0) recover_cheirality_kernel<<<dim3((max_n + 127) / 128, 4, nseq), 128, 0, stream>>>(a);
    recover_pick_kernel<<<nseq, 32, 0, stream>>>(a);
    ctx->launches += max_n > 0 ? 3 : 2;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

extern "C" int b200vo_recover_pose(b200vo_ctx* ctx, const double E[9], const float* p1, const float* p2, int n,
                                   const double K[9], double distance_thresh, double R[9], double t[3], uint8_t* mask,
                                   int* n_good)
{
    if (!ctx || !E || !K || !R || !t || !n_good || n < 0 || (n > 0 && (!p1 || !p2 || !mask))) return B200VO_E_BADARG;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    RecArgs a{};
    VO_TRY(vo_intrinsics_uniform(ctx, K, VO_BOOT_EMAT_THR, 1, &a.intr));   // the batch of one
    a.dist = distance_thresh; a.cap = n;
    const int nn = n > 0 ? n : 1;
    const size_t b_p = vo_align((size_t)nn * 8, 256), b_m = vo_align((size_t)4 * nn, 256), b_small = 512;
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[7], 2 * b_p + b_small + b_m + b_small));
    VO_TRY(vo_reserve_pinned(ctx, 2 * b_p + b_small + b_m + b_small));
    uint8_t* d = (uint8_t*)ctx->d_scratch[7].p;
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    // in: p1 | p2 | E[9], n   out: masks [4][n] | R|t [12], winner, count, good [4] | poses [4][12] (b_small bytes after the masks)
    if (n > 0) { memcpy(hp, p1, (size_t)n * 8); memcpy(hp + b_p, p2, (size_t)n * 8); }
    memcpy(hp + 2 * b_p, E, 72);
    memcpy(hp + 2 * b_p + 128, &n, 4);
    VO_CUDA(ctx, cudaMemcpyAsync(d, hp, 2 * b_p + b_small, cudaMemcpyHostToDevice, ctx->stream));
    a.p1 = (const float*)d; a.p2 = (const float*)(d + b_p);
    a.E = (const double*)(d + 2 * b_p); a.n = (const int*)(d + 2 * b_p + 128);
    uint8_t* dout = d + 2 * b_p + b_small;
    a.masks = dout;
    a.Rt = (double*)(dout + b_m); a.win = (int*)(dout + b_m + 96); a.good = (int*)(dout + b_m + 112);
    a.poses = (double*)(dout + b_m + 128);
    VO_TRY(vo_recover_pose_batch_launch(ctx, a, 1, n, ctx->stream));
    uint8_t* ho = hp + 2 * b_p + b_small;
    VO_CUDA(ctx, cudaMemcpyAsync(ho, dout, b_m + 128, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    const double* rt = (const double*)(ho + b_m);
    const int* w = (const int*)(ho + b_m + 96);
    for (int k = 0; k < 9; ++k) R[k] = rt[k];
    for (int k = 0; k < 3; ++k) t[k] = rt[9 + k];
    if (n > 0) memcpy(mask, ho + (size_t)w[0] * n, (size_t)n);
    *n_good = w[1];
    return 0;
}
