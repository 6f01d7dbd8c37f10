// C-ABI glue for cv2.solvePnPRansac(flags=SOLVEPNP_P3P) (reference VisualOdometryPipeLine.py:343).
#include "internal.cuh"
#include "pnp.cuh"

static int pnp_run(b200vo_ctx* ctx, const float* obj, const float* img, int n, const double K[9],
                   const int32_t* samples, int iters, float reproj_err, double conf, double rvec[3],
                   double tvec[3], int32_t* inliers, int* n_inliers, int* success, int32_t* counts_out,
                   int* winner_iter, int* iters_run)
{
    if (!ctx) return B200VO_E_BADARG;
    if (!obj || !img || !K || !rvec || !tvec || !inliers || !n_inliers || !success)
        return vo_set_err(ctx, B200VO_E_BADARG, "null pointer");
    if (n < 4)  // cv2: solvepnp.cpp CV_Assert(npoints >= 4 && ...)
        return vo_set_err(ctx, B200VO_E_BADARG, "npoints >= 4 && npoints == std::max(ipoints.checkVector(2, CV_32F), ipoints.checkVector(2, CV_64F))");
    if (iters < 1) iters = 1;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    PnpArgs a{};
    a.batch = 1; a.cap = n; a.iters = iters;
    VO_TRY(vo_intrinsics_uniform(ctx, K, VO_BOOT_EMAT_THR, 1, &a.intr));   // the batch of one
    a.thr_sq = (float)((double)reproj_err * (double)reproj_err);
    a.conf = conf;
    a.full_counts = counts_out != nullptr;
    a.n_raw = 8 * iters + 256;
    VO_TRY(vo_rng_table(ctx, a.n_raw, &a.rng_raw));
    // device layout: [obj | img | n | inliers | mask | pose | ok] + workspace
    const size_t b_obj = vo_align((size_t)n * 12, 256), b_img = vo_align((size_t)n * 8, 256), b_n = 256;
    const size_t b_inl = vo_align((size_t)n * 4, 256), b_mask = vo_align((size_t)n, 256), b_pose = 256, b_ok = 256;
    const size_t b_ws = vo_pnp_workspace_bytes(1, n, iters);
    const size_t in_bytes = b_obj + b_img + b_n;
    const size_t out_bytes = b_inl + b_mask + b_pose + b_ok;
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[1], in_bytes + out_bytes + b_ws));
    uint8_t* d = (uint8_t*)ctx->d_scratch[1].p;
    a.obj = (const float*)d; a.img = (const float*)(d + b_obj); a.n = (const int*)(d + b_obj + b_img);
    uint8_t* dout = d + in_bytes;
    a.inliers = (int*)dout; a.mask = dout + b_inl; a.pose = (double*)(dout + b_inl + b_mask);
    a.ok = dout + b_inl + b_mask + b_pose;
    vo_pnp_carve_workspace(a, dout + out_bytes);
    // host staging: inputs then outputs (+ small results)
    const size_t b_small = 256;
    const size_t b_cnt = counts_out ? vo_align((size_t)iters * 4, 256) : 0;
    VO_TRY(vo_reserve_pinned(ctx, in_bytes + out_bytes + b_small + b_cnt + (samples ? (size_t)iters * 16 : 0)));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    memcpy(hp, obj, (size_t)n * 12);
    memcpy(hp + b_obj, img, (size_t)n * 8);
    *(int*)(hp + b_obj + b_img) = n;
    VO_CUDA(ctx, cudaMemcpyAsync(d, hp, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
    if (samples) {
        uint8_t* hs = hp + in_bytes + out_bytes + b_small + b_cnt;
        memcpy(hs, samples, (size_t)iters * 16);
        VO_CUDA(ctx, cudaMemcpyAsync(a.samples, hs, (size_t)iters * 16, cudaMemcpyHostToDevice, ctx->stream));
    }
    VO_TRY(vo_pnp_launch(ctx, a, samples == nullptr, ctx->stream));
    uint8_t* ho = hp + in_bytes;
    VO_CUDA(ctx, cudaMemcpyAsync(ho, dout, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    int* hsmall = (int*)(ho + out_bytes);
    VO_CUDA(ctx, cudaMemcpyAsync(hsmall, a.winner, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaMemcpyAsync(hsmall + 1, a.iters_run, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaMemcpyAsync(hsmall + 2, a.n_inliers, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaMemcpyAsync(hsmall + 3, a.flags, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (counts_out)
        VO_CUDA(ctx, cudaMemcpyAsync(ho + out_bytes + b_small, a.counts, (size_t)iters * 4, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    if (hsmall[3] & 1) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "RNG table exhausted while drawing subsets (n=%d)", n);
    const int ok = ho[b_inl + b_mask + b_pose];
    const int m = hsmall[2];
    *success = ok;
    *n_inliers = ok ? m : 0;
    if (winner_iter) *winner_iter = hsmall[0];
    if (iters_run) *iters_run = hsmall[1];
    if (counts_out) memcpy(counts_out, ho + out_bytes + b_small, (size_t)iters * 4);
    if (ok) {
        memcpy(inliers, ho, (size_t)m * 4);
        const double* pose = (const double*)(ho + b_inl + b_mask);
        for (int k = 0; k < 3; ++k) { rvec[k] = pose[k]; tvec[k] = pose[3 + k]; }
    }
    return 0;
}

extern "C" int b200vo_solve_pnp_ransac_p3p(b200vo_ctx* ctx, const float* obj, const float* img, int n,
                                           const double K[9], int iters, float reproj_err, double conf,
                                           double rvec[3], double tvec[3], int32_t* inliers, int* n_inliers,
                                           int* success)
{
    return pnp_run(ctx, obj, img, n, K, nullptr, iters, reproj_err, conf, rvec, tvec, inliers, n_inliers, success,
                   nullptr, nullptr, nullptr);
}

extern "C" int b200vo_solve_pnp_ransac_p3p_samples(b200vo_ctx* ctx, const float* obj, const float* img, int n,
                                                   const double K[9], const int32_t* samples, int iters,
                                                   float reproj_err, double conf, double rvec[3], double tvec[3],
                                                   int32_t* inliers, int* n_inliers, int* success,
                                                   int32_t* counts_out, int* winner_iter, int* iters_run)
{
    return pnp_run(ctx, obj, img, n, K, samples, iters, reproj_err, conf, rvec, tvec, inliers, n_inliers, success,
                   counts_out, winner_iter, iters_run);
}

// Device-pointer form (SURVEY 8b `_dev`): obj_dev float32 (n,3), img_dev float32 (n,2) in device memory; pose_dev double[6]
// (rvec | tvec), inliers_dev int32 (n) ascending, n_inliers_dev int32[1], success_dev uint8[1] are written on the device.
// Asynchronous on the ctx stream.
__global__ void pnp_export_kernel(const int* __restrict__ n_inl, const uint8_t* __restrict__ ok, int32_t* __restrict__ n_out)
{
    *n_out = *ok ? *n_inl : 0;
}

extern "C" int b200vo_solve_pnp_ransac_p3p_dev(b200vo_ctx* ctx, const float* obj_dev, const float* img_dev, int n, const double K[9],
                                               int iters, float reproj_err, double conf, double* pose_dev, int32_t* inliers_dev,
                                               int32_t* n_inliers_dev, uint8_t* success_dev)
{
    if (!ctx) return B200VO_E_BADARG;
    if (!obj_dev || !img_dev || !K || !pose_dev || !inliers_dev || !n_inliers_dev || !success_dev)
        return vo_set_err(ctx, B200VO_E_BADARG, "null pointer");
    if (n < 4)  // cv2: solvepnp.cpp CV_Assert(npoints >= 4 && ...)
        return vo_set_err(ctx, B200VO_E_BADARG, "npoints >= 4 && npoints == std::max(ipoints.checkVector(2, CV_32F), ipoints.checkVector(2, CV_64F))");
    if (iters < 1) iters = 1;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    PnpArgs a{};
    a.batch = 1; a.cap = n; a.iters = iters;
    VO_TRY(vo_intrinsics_uniform(ctx, K, VO_BOOT_EMAT_THR, 1, &a.intr));   // the batch of one
    a.thr_sq = (float)((double)reproj_err * (double)reproj_err);
    a.conf = conf;
    a.n_raw = 8 * iters + 256;
    VO_TRY(vo_rng_table(ctx, a.n_raw, &a.rng_raw));
    const size_t b_mask = vo_align((size_t)n, 256), b_ws = vo_pnp_workspace_bytes(1, n, iters);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[1], 256 + b_mask + b_ws));
    uint8_t* d = (uint8_t*)ctx->d_scratch[1].p;
    a.obj = obj_dev; a.img = img_dev; a.n = (const int*)d;
    a.mask = d + 256;
    a.inliers = inliers_dev; a.pose = pose_dev; a.ok = success_dev;
    vo_pnp_carve_workspace(a, d + 256 + b_mask);
    VO_CUDA(ctx, cudaMemcpyAsync(d, &n, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));   // pageable source: staged before the call returns
    VO_TRY(vo_pnp_launch(ctx, a, true, ctx->stream));
    pnp_export_kernel<<<1, 1, 0, ctx->stream>>>(a.n_inliers, a.ok, n_inliers_dev);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// Measurement aid (benchmarks/pose_phases.py): the device-pointer PnP call with the fused kernel's phase stamps
// (clock64 of thread 0 at the phase boundaries listed in pnp.cu) copied to clk_host[16] after a synchronisation.
extern "C" int b200vo_debug_pose_phases(b200vo_ctx* ctx, const float* obj_dev, const float* img_dev, int n, const double K[9], int iters,
                                        float reproj_err, double conf, long long* clk_host, float* kernel_ms)
{
    if (!ctx || !obj_dev || !img_dev || !K || !clk_host || n < 4) return B200VO_E_BADARG;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    PnpArgs a{};
    a.batch = 1; a.cap = n; a.iters = iters < 1 ? 1 : iters;
    VO_TRY(vo_intrinsics_uniform(ctx, K, VO_BOOT_EMAT_THR, 1, &a.intr));   // the batch of one
    a.thr_sq = (float)((double)reproj_err * (double)reproj_err);
    a.conf = conf;
    a.n_raw = 8 * a.iters + 256;
    VO_TRY(vo_rng_table(ctx, a.n_raw, &a.rng_raw));
    const size_t b_mask = vo_align((size_t)n, 256), b_inl = vo_align((size_t)n * 4, 256), b_ws = vo_pnp_workspace_bytes(1, n, a.iters);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[1], 1024 + b_mask + b_inl + b_ws));
    uint8_t* d = (uint8_t*)ctx->d_scratch[1].p;
    a.obj = obj_dev; a.img = img_dev; a.n = (const int*)d;
    a.pose = (double*)(d + 64); a.ok = d + 128; a.phase_clk = (long long*)(d + 256);
    a.mask = d + 1024; a.inliers = (int*)(d + 1024 + b_mask);
    vo_pnp_carve_workspace(a, d + 1024 + b_mask + b_inl);
    VO_CUDA(ctx, cudaMemsetAsync(d, 0, 1024, ctx->stream));
    VO_CUDA(ctx, cudaMemcpyAsync(d, &n, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    if (!vo_pnp_fused_ok(a, true)) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "the fused pose kernel is not in use for this size");
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    VO_TRY(vo_pnp_launch(ctx, a, true, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaMemcpyAsync(clk_host, a.phase_clk, 16 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (kernel_ms) cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1);
    return 0;
}

