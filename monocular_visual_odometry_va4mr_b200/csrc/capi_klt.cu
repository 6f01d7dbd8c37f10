// C-ABI glue for the tracker: cv2.calcOpticalFlowPyrLK drop-in (reference
// VisualOdometryPipeLine.py:281,287), in stateless and frame-slot form.
#include "internal.cuh"

static int klt_check_args(b200vo_ctx* ctx, int rows, int cols, int win_w, int win_h, int max_level, int flags)
{
    if (!ctx) return B200VO_E_BADARG;
    if (max_level < 0 || win_w <= 2 || win_h <= 2)  // cv2: lkpyramid.cpp CV_Assert(maxLevel >= 0 && winSize.width > 2 && winSize.height > 2)
        return vo_set_err(ctx, B200VO_E_BADARG, "maxLevel >= 0 && winSize.width > 2 && winSize.height > 2");
    if (rows <= 0 || cols <= 0) return vo_set_err(ctx, B200VO_E_BADARG, "empty image");
    if (flags != 0) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "flags != 0 (OPTFLOW_USE_INITIAL_FLOW / LK_GET_MIN_EIGENVALS) not implemented");
    if (win_w >= VO_BORDER || win_h >= VO_BORDER)
        return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "winSize > %d not implemented", VO_BORDER - 1);
    if (cols <= win_w || rows <= win_h)
        return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "image not larger than the window");
    return 0;
}

static KltParams make_params(int win_w, int win_h, int crit_type, int crit_max_count, double crit_eps, double min_eig)
{
    KltParams kp;
    kp.win_w = win_w;
    kp.win_h = win_h;
    // cv2 (lkpyramid.cpp): COUNT -> clamp(maxCount, 0, 100) else 30; EPS -> clamp(eps, 0, 10) else 0.01; eps *= eps
    kp.max_count = (crit_type & 1) ? (crit_max_count < 0 ? 0 : crit_max_count > 100 ? 100 : crit_max_count) : 30;
    double eps = (crit_type & 2) ? (crit_eps < 0 ? 0 : crit_eps > 10 ? 10 : crit_eps) : 0.01;
    kp.eps_sq = eps * eps;
    kp.min_eig_thr = (float)min_eig;
    return kp;
}

static int upload_into_slot(b200vo_ctx* ctx, int slot, int stage_idx, const uint8_t* img, int rows, int cols,
                            size_t step, int win_w, int win_h, int max_level)
{
    FrameSlot& fs = ctx->slots[slot];
    const int levels = vo_pyr_levels(cols, rows, win_w, win_h, max_level);
    PyrGeom g;
    vo_pyr_geom(rows, cols, levels, &g);
    VO_TRY(vo_reserve(ctx, fs.slab, g.slab_bytes));
    const size_t raw_bytes = (size_t)rows * cols;
    VO_TRY(vo_reserve(ctx, ctx->d_stage_img[stage_idx], raw_bytes));
    // pinned staging: [stage_idx * raw_bytes]
    VO_TRY(vo_reserve_pinned(ctx, 2 * vo_align(raw_bytes, 256) + (1 << 20)));
    uint8_t* hp = (uint8_t*)ctx->h_pin + stage_idx * vo_align(raw_bytes, 256);
    if (step == (size_t)cols) memcpy(hp, img, raw_bytes);
    else for (int y = 0; y < rows; ++y) memcpy(hp + (size_t)y * cols, img + (size_t)y * step, (size_t)cols);
    VO_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage_img[stage_idx].p, hp, raw_bytes, cudaMemcpyHostToDevice, ctx->stream));
    VO_TRY(vo_build_pyramids(ctx, (const uint8_t*)ctx->d_stage_img[stage_idx].p, raw_bytes, rows, cols, g,
                             (uint8_t*)fs.slab.p, g.slab_bytes, 1, ctx->stream));
    fs.geom = g;
    fs.rows = rows;
    fs.cols = cols;
    fs.valid = true;
    return 0;
}

static int klt_on_slots(b200vo_ctx* ctx, int prev_slot, int next_slot, const float* prev_pts, int n,
                        const KltParams& kp, int max_level, float* next_pts, uint8_t* status, float* err,
                        size_t pin_off)
{
    FrameSlot& fp = ctx->slots[prev_slot];
    FrameSlot& fn = ctx->slots[next_slot];
    if (!fp.valid || !fn.valid) return vo_set_err(ctx, B200VO_E_BADARG, "frame slot not uploaded");
    if (fp.rows != fn.rows || fp.cols != fn.cols)
        return vo_set_err(ctx, B200VO_E_BADARG, "prevPyr[level].size() == nextPyr[level].size()");
    const int levels = vo_pyr_levels(fp.cols, fp.rows, kp.win_w, kp.win_h, max_level);
    if (levels > fp.geom.levels || levels > fn.geom.levels)
        return vo_set_err(ctx, B200VO_E_BADARG, "slot pyramid has fewer levels than this call needs");
    PyrGeom g = fp.geom;
    g.levels = levels;
    // device scratch: pts | next | err | status
    const size_t b_pts = vo_align((size_t)n * 8, 256), b_err = vo_align((size_t)n * 4, 256), b_st = vo_align((size_t)n, 256);
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[0], 2 * b_pts + b_err + b_st));
    uint8_t* d = (uint8_t*)ctx->d_scratch[0].p;
    float* d_pts = (float*)d;
    float* d_next = (float*)(d + b_pts);
    float* d_err = (float*)(d + 2 * b_pts);
    uint8_t* d_st = d + 2 * b_pts + b_err;
    VO_TRY(vo_reserve_pinned(ctx, pin_off + 2 * b_pts + b_err + b_st));
    uint8_t* hp = (uint8_t*)ctx->h_pin + pin_off;
    memcpy(hp, prev_pts, (size_t)n * 8);
    VO_CUDA(ctx, cudaMemcpyAsync(d_pts, hp, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    const KltPointSet set{n, nullptr, d_pts, d_next, d_st, d_err};
    VO_TRY(vo_klt_launch2(ctx, g, (const uint8_t*)fp.slab.p, 0, (const uint8_t*)fn.slab.p, 0, 1, &set, 1, n, kp, ctx->stream));
    // one D2H of next|err|status (contiguous on the device)
    VO_CUDA(ctx, cudaMemcpyAsync(hp + b_pts, d_next, b_pts + b_err + b_st, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    memcpy(next_pts, hp + b_pts, (size_t)n * 8);
    memcpy(err, hp + 2 * b_pts, (size_t)n * 4);
    memcpy(status, hp + 2 * b_pts + b_err, (size_t)n);
    return 0;
}

extern "C" int b200vo_calc_optical_flow_pyr_lk(b200vo_ctx* ctx, const uint8_t* prev, const uint8_t* next,
                                               int rows, int cols, size_t prev_step, size_t next_step,
                                               const float* prev_pts, int n, int win_w, int win_h,
                                               int max_level, int crit_type, int crit_max_count,
                                               double crit_eps, int flags, double min_eig_thr,
                                               float* next_pts, uint8_t* status, float* err)
{
    VO_TRY(klt_check_args(ctx, rows, cols, win_w, win_h, max_level, flags));
    if (!prev || !next || (n > 0 && (!prev_pts || !next_pts || !status || !err)))
        return vo_set_err(ctx, B200VO_E_BADARG, "null pointer");
    if (n < 0) return vo_set_err(ctx, B200VO_E_BADARG, "npoints >= 0");
    if (n == 0) return 0;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const int s0 = B200VO_MAX_SLOTS, s1 = B200VO_MAX_SLOTS + 1;  // internal slots
    VO_TRY(upload_into_slot(ctx, s0, 0, prev, rows, cols, prev_step, win_w, win_h, max_level));
    VO_TRY(upload_into_slot(ctx, s1, 1, next, rows, cols, next_step, win_w, win_h, max_level));
    KltParams kp = make_params(win_w, win_h, crit_type, crit_max_count, crit_eps, min_eig_thr);
    const size_t pin_off = 2 * vo_align((size_t)rows * cols, 256);
    return klt_on_slots(ctx, s0, s1, prev_pts, n, kp, max_level, next_pts, status, err, pin_off);
}

// pyramid of a DEVICE-resident image into an internal slot (no host staging)
static int build_slot_from_device(b200vo_ctx* ctx, int slot, int stage_idx, const uint8_t* img_dev, int rows, int cols, size_t step,
                                  int win_w, int win_h, int max_level)
{
    FrameSlot& fs = ctx->slots[slot];
    const int levels = vo_pyr_levels(cols, rows, win_w, win_h, max_level);
    PyrGeom g;
    vo_pyr_geom(rows, cols, levels, &g);
    VO_TRY(vo_reserve(ctx, fs.slab, g.slab_bytes));
    const size_t raw_bytes = (size_t)rows * cols;
    const uint8_t* raw = img_dev;
    if (step != (size_t)cols) {     // pitched view: pack the rows first
        VO_TRY(vo_reserve(ctx, ctx->d_stage_img[stage_idx], raw_bytes));
        VO_CUDA(ctx, cudaMemcpy2DAsync(ctx->d_stage_img[stage_idx].p, (size_t)cols, img_dev, step, (size_t)cols, (size_t)rows,
                                       cudaMemcpyDeviceToDevice, ctx->stream));
        raw = (const uint8_t*)ctx->d_stage_img[stage_idx].p;
    }
    VO_TRY(vo_build_pyramids(ctx, raw, raw_bytes, rows, cols, g, (uint8_t*)fs.slab.p, g.slab_bytes, 1, ctx->stream));
    fs.geom = g; fs.rows = rows; fs.cols = cols; fs.valid = true;
    return 0;
}

// Device-pointer form of b200vo_calc_optical_flow_pyr_lk (SURVEY 8b `_dev`): images, points and results stay in device
// memory; asynchronous on the ctx stream (pair with b200vo_sync).
extern "C" int b200vo_calc_optical_flow_pyr_lk_dev(b200vo_ctx* ctx, const uint8_t* prev_dev, const uint8_t* next_dev, int rows, int cols,
                                                   size_t prev_step, size_t next_step, const float* prev_pts_dev, int n, int win_w,
                                                   int win_h, int max_level, int crit_type, int crit_max_count, double crit_eps,
                                                   int flags, double min_eig_thr, float* next_pts_dev, uint8_t* status_dev,
                                                   float* err_dev)
{
    VO_TRY(klt_check_args(ctx, rows, cols, win_w, win_h, max_level, flags));
    if (!prev_dev || !next_dev || (n > 0 && (!prev_pts_dev || !next_pts_dev || !status_dev)))
        return vo_set_err(ctx, B200VO_E_BADARG, "null pointer");
    if (n < 0) return vo_set_err(ctx, B200VO_E_BADARG, "npoints >= 0");
    if (prev_step < (size_t)cols || next_step < (size_t)cols) return vo_set_err(ctx, B200VO_E_BADARG, "step < cols");
    if (n == 0) return 0;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    const int s0 = B200VO_MAX_SLOTS, s1 = B200VO_MAX_SLOTS + 1;  // internal slots
    VO_TRY(build_slot_from_device(ctx, s0, 0, prev_dev, rows, cols, prev_step, win_w, win_h, max_level));
    VO_TRY(build_slot_from_device(ctx, s1, 1, next_dev, rows, cols, next_step, win_w, win_h, max_level));
    const KltParams kp = make_params(win_w, win_h, crit_type, crit_max_count, crit_eps, min_eig_thr);
    const FrameSlot& fp = ctx->slots[s0];
    const KltPointSet set{n, nullptr, prev_pts_dev, next_pts_dev, status_dev, err_dev};
    return vo_klt_launch2(ctx, fp.geom, (const uint8_t*)fp.slab.p, 0, (const uint8_t*)ctx->slots[s1].slab.p, 0, 1, &set, 1, n, kp,
                          ctx->stream);
}

extern "C" int b200vo_frame_upload(b200vo_ctx* ctx, int slot, const uint8_t* img, int rows, int cols,
                                   size_t step, int win_w, int win_h, int max_level)
{
    VO_TRY(klt_check_args(ctx, rows, cols, win_w, win_h, max_level, 0));
    if (slot < 0 || slot >= B200VO_MAX_SLOTS || !img) return vo_set_err(ctx, B200VO_E_BADARG, "bad slot / null image");
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_TRY(upload_into_slot(ctx, slot, 0, img, rows, cols, step, win_w, win_h, max_level));
    // the pinned staging area is reused by the next call: make the upload complete before returning
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

extern "C" int b200vo_klt_slots(b200vo_ctx* ctx, int prev_slot, int next_slot, const float* prev_pts, int n,
                                int win_w, int win_h, int max_level, int crit_type, int crit_max_count,
                                double crit_eps, int flags, double min_eig_thr,
                                float* next_pts, uint8_t* status, float* err)
{
    if (!ctx) return B200VO_E_BADARG;
    if (prev_slot < 0 || prev_slot >= B200VO_MAX_SLOTS || next_slot < 0 || next_slot >= B200VO_MAX_SLOTS)
        return vo_set_err(ctx, B200VO_E_BADARG, "bad slot");
    VO_TRY(klt_check_args(ctx, ctx->slots[prev_slot].rows ? ctx->slots[prev_slot].rows : 1,
                          ctx->slots[prev_slot].cols ? ctx->slots[prev_slot].cols : 1, win_w, win_h, max_level, flags));
    if (n < 0 || (n > 0 && (!prev_pts || !next_pts || !status || !err))) return vo_set_err(ctx, B200VO_E_BADARG, "bad points");
    if (n == 0) return 0;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    KltParams kp = make_params(win_w, win_h, crit_type, crit_max_count, crit_eps, min_eig_thr);
    return klt_on_slots(ctx, prev_slot, next_slot, prev_pts, n, kp, max_level, next_pts, status, err, 0);
}

extern "C" int b200vo_frame_download_level(b200vo_ctx* ctx, int slot, int level, uint8_t* out, int* w, int* h,
                                           int* n_levels)
{
    if (!ctx || slot < 0 || slot >= B200VO_MAX_SLOTS + 2) return B200VO_E_BADARG;
    FrameSlot& fs = ctx->slots[slot];
    if (!fs.valid) return vo_set_err(ctx, B200VO_E_BADARG, "frame slot not uploaded");
    if (n_levels) *n_levels = fs.geom.levels;
    if (level < 0 || level >= fs.geom.levels) return vo_set_err(ctx, B200VO_E_BADARG, "no such level");
    if (w) *w = fs.geom.w[level];
    if (h) *h = fs.geom.h[level];
    if (!out) return 0;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaMemcpy2DAsync(out, (size_t)fs.geom.w[level], (uint8_t*)fs.slab.p + fs.geom.off[level],
                                   (size_t)fs.geom.pitch[level], (size_t)fs.geom.w[level], (size_t)fs.geom.h[level],
                                   cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
