// The whole per-frame loop of the reference (VisualOdometryPipeLine.py `continuous_operation` :326-373, with the data
// flow of tests/mini_vo.py `MiniVO.step`) for a batch of independent sequences.  The VO state of every sequence --
// landmarks, candidates, pose history -- stays in device memory; one step is the batch object's tracker + pose chain
// (batch.cu), batched goodFeaturesToTrack (gftt.cu), the batched triangulation and distance filter (landmarks.cu) and
// three small kernels of this file that do what the reference does with numpy between those calls:
//   commit     stop decisions, inlier landmarks, tracked candidates, (R_CW | t_CW) from rvec | tvec
//   merge      append the triangulated landmarks, keep the too_short_baseline candidates
//   append     append the corners that pass the distance filter as candidates, append the pose
// Between steps the state lives in one canonical set of arrays; every kernel that rewrites a range reads it from a
// scratch copy (the tracker output, the compacted PnP input, the candidates after the status filter), so no kernel
// reads and writes the same slots.
#include "batch.cuh"
#include "landmarks.cuh"
#include "mathdev.cuh"
#include "pnp.cuh"

#define LOOP_T 256

struct LoopOut {   // per-sequence results of a step: the packed block of b200vo_loop_step or the caller's device arrays
    int* status; int* n_inl; int* n_lm; int* n_cand; double* pose;
};

struct LoopDev {   // kernel view of the state and of the step's scratch (device memory)
    int L, C, P, G;            // capacities: landmarks, candidates, poses; G = corner slots per sequence of the detector output
    // state
    float* lm; float* lm_kp;                   // [batch][L][3], [batch][L][2]
    float* keys; float* fkeys; int* fpose;     // [batch][C][2], [batch][C][2], [batch][C]
    double* poses;                             // [batch][P][12]  R_CW row-major | t_CW
    int* n_lm; int* n_cand; int* n_poses; int* status;
    int* trk_lm; int* trk_cand;                // points the next step's trackers see (0: sequence stopped / candidates not tracked)
    // scratch of one step
    float* lm_next; uint8_t* lm_status; float* cand_next; uint8_t* cand_status;
    double* pose6; uint8_t* pnp_ok; uint8_t* inl_mask; int* n_inl;
    const float* c_obj; const float* c_img; const int* c_n; const int* inliers;   // compacted PnP input and its inliers
    float* keys_b; float* fkeys_b; int* fpose_b; int* n_cand_b;                   // candidates after the status filter
    double* cur_pose;                          // [batch][12]
    int* tri_n;                                // candidates handed to the triangulation (0: it does not run)
    uint8_t* keep; float* new_lm; float* new_kp; int* n_new;                      // its outputs ([batch][C]...)
    const float* corners; const int* gftt_small;                                  // detector output
    int* n_corner; uint8_t* valid;             // corners per sequence, distance-filter result [batch][G]
};

// Ordered compaction of [0, n) by one CTA of LOOP_T threads: emit(i, o) for every i with keep(i), o = its rank among
// the kept ones (what numpy's boolean indexing does).  Returns the count to every thread.
template <class Keep, class Emit>
__device__ __forceinline__ int cta_compact(int n, Keep keep, Emit emit)
{
    __shared__ int s_warp[LOOP_T / 32];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < n; base += LOOP_T) {
        const int i = base + threadIdx.x;
        const bool k = i < n && keep(i);
        const unsigned bm = __ballot_sync(0xffffffffu, k);
        if (lane == 0) s_warp[warp] = __popc(bm);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += s_warp[w];
        if (k) emit(i, off + __popc(bm & ((1u << lane) - 1)));
        __syncthreads();
        if (threadIdx.x == 0) {
            int tot = 0;
            for (int w = 0; w < LOOP_T / 32; ++w) tot += s_warp[w];
            s_base += tot;
        }
        __syncthreads();
    }
    const int r = s_base;
    __syncthreads();
    return r;
}

// Steps 3-5 of MiniVO.step and the status filter of step 2: one CTA per sequence.
__global__ void __launch_bounds__(LOOP_T)
loop_commit_kernel(LoopDev d, LoopOut out)
{
    __shared__ int s_code;
    const int s = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) {
        int code = d.status[s];
        if (code == B200VO_LOOP_OK) {
            if (d.c_n[s] < 8) code = B200VO_LOOP_FEW_POINTS;
            else if (!d.pnp_ok[s]) code = B200VO_LOOP_PNP_FAILED;
            else if (d.gftt_small[s * VO_GFTT_SMALL + 1] > VO_GFTT_BATCH_CAP) code = B200VO_LOOP_DETECT_LIMIT;
            else if (d.n_poses[s] >= d.P) code = B200VO_LOOP_OVERFLOW;
            d.status[s] = code;
        }
        s_code = code;
        if (code != B200VO_LOOP_OK) { d.tri_n[s] = 0; d.n_corner[s] = 0; }
    }
    __syncthreads();
    if (s_code != B200VO_LOOP_OK) return;   // a sequence that stops keeps the state it had before the step
    if (tid == 0) {   // R_WC = Rodrigues(rvec), R_CW = R_WC^T, t_CW = -R_WC^T tvec (:354-355)
        const double* rt = d.pose6 + 6 * s;
        double R[9], cw[12];
        vo::rodrigues_to_R(rt, R);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) cw[3 * i + j] = R[3 * j + i];
        for (int i = 0; i < 3; ++i) cw[9 + i] = -R[i] * rt[3] + -R[3 + i] * rt[4] + -R[6 + i] * rt[5];
        double* hist = d.poses + ((size_t)s * d.P + d.n_poses[s]) * 12;   // appended by loop_append_kernel
        for (int k = 0; k < 12; ++k) { d.cur_pose[12 * s + k] = cw[k]; hist[k] = cw[k]; out.pose[12 * s + k] = cw[k]; }
        out.n_inl[s] = d.n_inl[s];
        d.n_corner[s] = d.gftt_small[s * VO_GFTT_SMALL + 2];
    }
    // the inliers of the tracked landmarks, in order (:346-350)
    const int m = d.n_inl[s];
    const size_t lo = (size_t)s * d.L;
    for (int k = tid; k < m; k += LOOP_T) {
        const size_t j = lo + d.inliers[lo + k];
        d.lm[3 * (lo + k)] = d.c_obj[3 * j]; d.lm[3 * (lo + k) + 1] = d.c_obj[3 * j + 1]; d.lm[3 * (lo + k) + 2] = d.c_obj[3 * j + 2];
        d.lm_kp[2 * (lo + k)] = d.c_img[2 * j]; d.lm_kp[2 * (lo + k) + 1] = d.c_img[2 * j + 1];
    }
    // the tracked candidates, in order (:287-289); untracked candidate sets (n <= 1) pass unchanged
    const size_t co = (size_t)s * d.C;
    const bool tracked = d.trk_cand[s] > 0;
    const float* kin = tracked ? d.cand_next : d.keys;
    const int nc = cta_compact(d.n_cand[s], [&](int i) { return !tracked || d.cand_status[co + i] == 1; },
                               [&](int i, int o) {
                                   d.keys_b[2 * (co + o)] = kin[2 * (co + i)]; d.keys_b[2 * (co + o) + 1] = kin[2 * (co + i) + 1];
                                   d.fkeys_b[2 * (co + o)] = d.fkeys[2 * (co + i)]; d.fkeys_b[2 * (co + o) + 1] = d.fkeys[2 * (co + i) + 1];
                                   d.fpose_b[co + o] = d.fpose[co + i];
                               });
    if (tid == 0) {
        d.n_lm[s] = m;
        d.n_cand_b[s] = nc;
        d.tri_n[s] = nc > 1 ? nc : 0;   // the reference triangulates only when more than one candidate is left (:371)
    }
}

// Step 6 after the triangulation kernels: append the new landmarks, keep the too_short_baseline candidates (:206).
__global__ void __launch_bounds__(LOOP_T)
loop_merge_kernel(LoopDev d)
{
    const int s = blockIdx.x, tid = threadIdx.x;
    if (d.status[s] != B200VO_LOOP_OK) return;   // written by this kernel only by thread 0, after every read below
    const bool ran = d.tri_n[s] > 0;
    const int nn = ran ? d.n_new[s] : 0, nl = d.n_lm[s];
    const bool fits = nl + nn <= d.L;
    const size_t lo = (size_t)s * d.L, co = (size_t)s * d.C;
    if (fits)
        for (int k = tid; k < nn; k += LOOP_T) {
            const size_t o = lo + nl + k;
            d.lm[3 * o] = d.new_lm[3 * (co + k)]; d.lm[3 * o + 1] = d.new_lm[3 * (co + k) + 1]; d.lm[3 * o + 2] = d.new_lm[3 * (co + k) + 2];
            d.lm_kp[2 * o] = d.new_kp[2 * (co + k)]; d.lm_kp[2 * o + 1] = d.new_kp[2 * (co + k) + 1];
        }
    const int nc = cta_compact(d.n_cand_b[s], [&](int i) { return !ran || d.keep[co + i] != 0; },
                               [&](int i, int o) {
                                   d.keys[2 * (co + o)] = d.keys_b[2 * (co + i)]; d.keys[2 * (co + o) + 1] = d.keys_b[2 * (co + i) + 1];
                                   d.fkeys[2 * (co + o)] = d.fkeys_b[2 * (co + i)]; d.fkeys[2 * (co + o) + 1] = d.fkeys_b[2 * (co + i) + 1];
                                   d.fpose[co + o] = d.fpose_b[co + i];
                               });
    if (tid == 0) {
        if (fits) d.n_lm[s] = nl + nn;
        else d.status[s] = B200VO_LOOP_OVERFLOW;
        d.n_cand[s] = nc;
    }
}

// Steps 7-8: append the corners that passed the distance filter (:258-268) and the pose; write the result block and
// the point counts the next step's trackers see.
__global__ void __launch_bounds__(LOOP_T)
loop_append_kernel(LoopDev d, LoopOut out)
{
    __shared__ int s_st;
    const int s = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) s_st = d.status[s];
    __syncthreads();
    if (s_st == B200VO_LOOP_OK) {
        const int nc = d.n_cand[s], np = d.n_poses[s];
        const size_t co = (size_t)s * d.C, go = (size_t)s * d.G;
        const int cnt = cta_compact(d.n_corner[s], [&](int i) { return d.valid[go + i] != 0; },
                                    [&](int i, int o) {
                                        if (nc + o >= d.C) return;
                                        const size_t q = co + nc + o;
                                        const float x = d.corners[2 * (go + i)], y = d.corners[2 * (go + i) + 1];
                                        d.keys[2 * q] = x; d.keys[2 * q + 1] = y;
                                        d.fkeys[2 * q] = x; d.fkeys[2 * q + 1] = y;
                                        d.fpose[q] = np;
                                    });
        if (tid == 0) {
            if (nc + cnt > d.C) { d.status[s] = B200VO_LOOP_OVERFLOW; s_st = B200VO_LOOP_OVERFLOW; }
            else { d.n_cand[s] = nc + cnt; d.n_poses[s] = np + 1; }
        }
    }
    if (tid == 0) {
        const int st = s_st, nl = d.n_lm[s], nc = d.n_cand[s];
        out.status[s] = st; out.n_lm[s] = nl; out.n_cand[s] = nc;
        if (st != B200VO_LOOP_OK) {
            out.n_inl[s] = 0;
            for (int k = 0; k < 12; ++k) out.pose[12 * s + k] = 0.0;
        }
        d.trk_lm[s] = st == B200VO_LOOP_OK ? nl : 0;
        d.trk_cand[s] = st == B200VO_LOOP_OK && nc > 1 ? nc : 0;   // the reference tracks candidates only when n > 1 (:286)
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
enum { CNT_LM, CNT_CAND, CNT_POSES, CNT_STATUS, CNT_TRK_LM, CNT_TRK_CAND, CNT_INL, CNT_CAND_B, CNT_TRI, CNT_NEW, CNT_CORNER,
       CNT_FLAGS, CNT_KINDS };

struct b200vo_loop {
    b200vo_ctx* ctx = nullptr;
    b200vo_batch* B = nullptr;   // pyramids, trackers, pose chain, streams
    b200vo_loop_cfg cfg{};
    int batch = 0;
    DevBuf mem;                  // state + scratch
    DevBuf res;                  // packed result block of b200vo_loop_step: pose_cw [batch][12] | status | n_inliers | n_lm | n_cand
    size_t res_bytes = 0;
    LoopDev d{};
    TriBatchArgs tri{};
    LoopOut res_out{};
};

extern "C" void b200vo_loop_destroy(b200vo_loop* lp)
{
    if (!lp) return;
    cudaSetDevice(lp->ctx->device);
    cudaStreamSynchronize(lp->ctx->stream);
    for (DevBuf* b : {&lp->mem, &lp->res}) if (b->p) cudaFree(b->p);
    b200vo_batch_destroy(lp->B);
    cudaGetLastError();
    delete lp;
}

extern "C" int b200vo_loop_create(b200vo_ctx* ctx, int batch, const b200vo_loop_cfg* cfg, b200vo_loop** out)
{
    if (!ctx || !cfg || !out || batch <= 0) return B200VO_E_BADARG;
    *out = nullptr;
    const b200vo_batch_cfg& bc = cfg->batch;
    if (cfg->max_frames < 2 || bc.max_candidates < 2 || cfg->max_corners <= 0 || !(cfg->quality_level > 0) || !(cfg->feature_min_dist >= 1))
        return vo_set_err(ctx, B200VO_E_BADARG, "the loop needs max_frames >= 2, max_candidates >= 2, max_corners > 0, "
                                                "quality_level > 0 and feature_min_dist >= 1");
    b200vo_batch* B = nullptr;
    VO_TRY(b200vo_batch_create(ctx, batch, &bc, &B));
    b200vo_loop* lp = new b200vo_loop();
    lp->ctx = ctx; lp->B = B; lp->cfg = *cfg; lp->batch = batch;
    LoopDev& d = lp->d;
    const int L = bc.max_landmarks, C = bc.max_candidates, P = cfg->max_frames;
    d.L = L; d.C = C; d.P = P;
    d.G = (int)(vo_align((size_t)cfg->max_corners * 8, 256) / 8);   // the detector's per-image output stride
    const size_t nb = batch, nl = nb * L, nc = nb * C;
    const size_t sizes[] = {nl * 12, nl * 8, nc * 8, nc * 8, nc * 4, nb * P * 96, (size_t)CNT_KINDS * nb * 4,
                            nl * 8, nl, nc * 8, nc, nb * 48, nb, nl,
                            nc * 8, nc * 8, nc * 4, nb * 96, nc, nc * 12, nc * 12, nc * 8, nb * d.G};
    size_t total = 0;
    for (size_t b : sizes) total += vo_align(b, 256);
    int rc = vo_reserve(ctx, lp->mem, total);
    lp->res_bytes = nb * 96 + 4 * nb * 4;
    if (!rc) rc = vo_reserve(ctx, lp->res, lp->res_bytes);
    if (!rc) rc = vo_reserve(ctx, B->gftt_ws, vo_gftt_batch_workspace(bc.rows, bc.cols, batch, cfg->max_corners));
    if (rc) { b200vo_loop_destroy(lp); return rc; }
    uint8_t* p = (uint8_t*)lp->mem.p;
    int k = 0;
    auto take = [&]() { uint8_t* r = p; p += vo_align(sizes[k++], 256); return (void*)r; };
    d.lm = (float*)take(); d.lm_kp = (float*)take(); d.keys = (float*)take(); d.fkeys = (float*)take(); d.fpose = (int*)take();
    d.poses = (double*)take();
    int* cnt = (int*)take();
    d.lm_next = (float*)take(); d.lm_status = (uint8_t*)take(); d.cand_next = (float*)take(); d.cand_status = (uint8_t*)take();
    d.pose6 = (double*)take(); d.pnp_ok = (uint8_t*)take(); d.inl_mask = (uint8_t*)take();
    d.keys_b = (float*)take(); d.fkeys_b = (float*)take(); d.fpose_b = (int*)take(); d.cur_pose = (double*)take();
    d.keep = (uint8_t*)take(); float* lm_slot = (float*)take(); d.new_lm = (float*)take(); d.new_kp = (float*)take();
    d.valid = (uint8_t*)take();
    d.n_lm = cnt + CNT_LM * nb; d.n_cand = cnt + CNT_CAND * nb; d.n_poses = cnt + CNT_POSES * nb; d.status = cnt + CNT_STATUS * nb;
    d.trk_lm = cnt + CNT_TRK_LM * nb; d.trk_cand = cnt + CNT_TRK_CAND * nb; d.n_inl = cnt + CNT_INL * nb;
    d.n_cand_b = cnt + CNT_CAND_B * nb; d.tri_n = cnt + CNT_TRI * nb; d.n_new = cnt + CNT_NEW * nb; d.n_corner = cnt + CNT_CORNER * nb;
    d.c_obj = B->c_obj; d.c_img = B->c_img; d.c_n = B->c_n; d.inliers = B->inliers;
    TriBatchArgs& t = lp->tri;
    vo_tri_common(t.common, bc.K, cfg->min_dist_landmarks, cfg->max_dist_landmarks, cfg->min_baseline_angle_deg, cfg->min_baseline_frames);
    t.cap = C; t.pose_cap = P;
    t.n = d.tri_n; t.n_poses = d.n_poses; t.cur = d.cur_pose;
    t.first_keys = d.fkeys_b; t.keys = d.keys_b; t.first_pose = d.fpose_b; t.poses = d.poses;
    t.keep = d.keep; t.lm_slot = lm_slot; t.out_lm = d.new_lm; t.out_kp = d.new_kp; t.n_new = d.n_new; t.flags = cnt + CNT_FLAGS * nb;
    uint8_t* r = (uint8_t*)lp->res.p;
    lp->res_out.pose = (double*)r;
    lp->res_out.status = (int*)(r + nb * 96);
    lp->res_out.n_inl = lp->res_out.status + nb; lp->res_out.n_lm = lp->res_out.n_inl + nb; lp->res_out.n_cand = lp->res_out.n_lm + nb;
    // every sequence starts IDLE with an empty state; the frames are blank until a sequence is loaded (the detector runs
    // over every image of the batch)
    std::vector<int> idle(batch, B200VO_LOOP_IDLE);
    cudaError_t e = cudaMemsetAsync(lp->mem.p, 0, total, ctx->stream);
    for (int s = 0; s < 3 && e == cudaSuccess; ++s) e = cudaMemsetAsync(B->slabs[s].p, 0, B->geom.slab_bytes * nb, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d.status, idle.data(), nb * 4, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaEventRecord(B->step_end_ev, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { b200vo_loop_destroy(lp); return vo_cuda_fail(ctx, e, "b200vo_loop_create: initial state"); }
    B->primed = true;
    *out = lp;
    return 0;
}

// one step of every sequence, enqueued on the ctx stream (the tracker and the pose chain use the batch object's streams
// and join it); frames_dev == nullptr: the oldest submitted frame set
static int loop_core(b200vo_loop* lp, const uint8_t* frames_dev, const LoopOut& o)
{
    b200vo_ctx* ctx = lp->ctx;
    b200vo_batch* B = lp->B;
    const b200vo_loop_cfg& c = lp->cfg;
    LoopDev& d = lp->d;
    const int nb = lp->batch;
    VO_TRY(batch_select_frames(B, frames_dev));
    VO_TRY(batch_track_pose_overlapped(B, frames_dev, d.lm_kp, d.lm, d.trk_lm, d.keys, d.trk_cand, d.lm_next, d.lm_status, d.cand_next,
                                       d.cand_status, d.pose6, d.pnp_ok, d.inl_mask, d.n_inl, nullptr));
    float* corners = nullptr;
    int* small = nullptr;
    VO_TRY(vo_gftt_batch_launch(ctx, (const uint8_t*)B->slabs[B->nxt].p + B->geom.off[0], B->geom.slab_bytes, B->geom.pitch[0],
                                c.batch.rows, c.batch.cols, nb, c.max_corners, c.quality_level, c.feature_min_dist, B->gftt_ws.p,
                                &corners, &small));
    d.corners = corners; d.gftt_small = small;
    loop_commit_kernel<<<nb, LOOP_T, 0, ctx->stream>>>(d, o);
    ctx->launches++;
    VO_TRY(vo_triangulate_batch_launch(ctx, lp->tri, nb, ctx->stream));
    loop_merge_kernel<<<nb, LOOP_T, 0, ctx->stream>>>(d);
    ctx->launches++;
    VO_TRY(vo_min_distance_batch_launch(ctx, nb, d.corners, d.n_corner, d.G, d.keys, d.n_cand, d.C, (float)c.feature_min_dist, d.valid,
                                        ctx->stream));
    loop_append_kernel<<<nb, LOOP_T, 0, ctx->stream>>>(d, o);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return batch_finish(B);
}

extern "C" int b200vo_loop_step_dev(b200vo_loop* lp, const uint8_t* frames_dev, int32_t* status_dev, int32_t* n_inliers_dev,
                                    int32_t* n_lm_dev, int32_t* n_cand_dev, double* pose_cw_dev)
{
    if (!lp || !status_dev || !n_inliers_dev || !n_lm_dev || !n_cand_dev || !pose_cw_dev) return B200VO_E_BADARG;
    VO_CUDA(lp->ctx, cudaSetDevice(lp->ctx->device));
    const LoopOut o{status_dev, n_inliers_dev, n_lm_dev, n_cand_dev, pose_cw_dev};
    return loop_core(lp, frames_dev, o);
}

extern "C" int b200vo_loop_step(b200vo_loop* lp, const uint8_t* frames, int32_t* status, int32_t* n_inliers, int32_t* n_lm,
                                int32_t* n_cand, double* pose_cw)
{
    if (!lp || !status || !n_inliers || !n_lm || !n_cand || !pose_cw) return B200VO_E_BADARG;
    b200vo_ctx* ctx = lp->ctx;
    b200vo_batch* B = lp->B;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const size_t nb = lp->batch, f_total = (size_t)lp->cfg.batch.rows * lp->cfg.batch.cols * nb;
    bool pinned = false;
    if (frames) {
        if (B->q_count > 0)
            return vo_set_err(ctx, B200VO_E_BADARG, "submitted frame sets are waiting: pass frames == NULL to consume them in order");
        cudaPointerAttributes at{};
        pinned = cudaPointerGetAttributes(&at, frames) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
    }
    const size_t staged = frames && !pinned ? vo_align(f_total, 256) : 0;
    VO_TRY(vo_reserve_pinned(ctx, staged + lp->res_bytes));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    const uint8_t* fdev = nullptr;
    if (frames) {   // the one upload of the step
        VO_TRY(vo_reserve(ctx, B->raw, f_total));
        if (!pinned) memcpy(hp, frames, f_total);
        VO_CUDA(ctx, cudaMemcpyAsync(B->raw.p, pinned ? frames : hp, f_total, cudaMemcpyHostToDevice, ctx->stream));
        fdev = (const uint8_t*)B->raw.p;
    }
    VO_TRY(loop_core(lp, fdev, lp->res_out));
    uint8_t* ho = hp + staged;   // the one read-back of the step
    VO_CUDA(ctx, cudaMemcpyAsync(ho, lp->res.p, lp->res_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    memcpy(pose_cw, ho, nb * 96);
    const int* ri = (const int*)(ho + nb * 96);
    memcpy(status, ri, nb * 4);
    memcpy(n_inliers, ri + nb, nb * 4);
    memcpy(n_lm, ri + 2 * nb, nb * 4);
    memcpy(n_cand, ri + 3 * nb, nb * 4);
    return 0;
}

extern "C" int b200vo_loop_submit_frames(b200vo_loop* lp, const uint8_t* frames)
{
    return lp ? batch_submit(lp->B, frames, false) : B200VO_E_BADARG;
}

extern "C" int b200vo_loop_submit_frames_dev(b200vo_loop* lp, const uint8_t* frames_dev)
{
    return lp ? batch_submit(lp->B, frames_dev, true) : B200VO_E_BADARG;
}

extern "C" int b200vo_loop_load(b200vo_loop* lp, int seq, const uint8_t* frame, const float* lm, const float* lm_kp, int n_lm,
                                const float* keys, const float* first_keys, const int32_t* first_pose, int n_cand,
                                const double* poses, int n_poses)
{
    if (!lp) return B200VO_E_BADARG;
    b200vo_ctx* ctx = lp->ctx;
    b200vo_batch* B = lp->B;
    const LoopDev& d = lp->d;
    if (seq < 0 || seq >= lp->batch) return vo_set_err(ctx, B200VO_E_BADARG, "seq = %d is outside [0, batch = %d)", seq, lp->batch);
    if (n_lm < 0 || n_lm > d.L) return vo_set_err(ctx, B200VO_E_BADARG, "n_lm = %d is outside [0, max_landmarks = %d]", n_lm, d.L);
    if (n_cand < 0 || n_cand > d.C) return vo_set_err(ctx, B200VO_E_BADARG, "n_cand = %d is outside [0, max_candidates = %d]", n_cand, d.C);
    if (n_poses < 1 || n_poses > d.P) return vo_set_err(ctx, B200VO_E_BADARG, "n_poses = %d is outside [1, max_frames = %d]", n_poses, d.P);
    if (!frame || !poses || (n_lm > 0 && (!lm || !lm_kp)) || (n_cand > 0 && (!keys || !first_keys || !first_pose)))
        return vo_set_err(ctx, B200VO_E_BADARG, "null array");
    for (int i = 0; i < n_cand; ++i)
        if (first_pose[i] < 0 || first_pose[i] >= n_poses)
            return vo_set_err(ctx, B200VO_E_BADARG, "first_pose[%d] = %d is outside [0, n_poses = %d)", i, first_pose[i], n_poses);
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // no step in flight reads the state
    cudaStream_t st = ctx->stream;
    const size_t fb = (size_t)lp->cfg.batch.rows * lp->cfg.batch.cols, sb = B->geom.slab_bytes;
    VO_TRY(vo_reserve(ctx, B->raw, fb));
    VO_CUDA(ctx, cudaMemcpyAsync(B->raw.p, frame, fb, cudaMemcpyHostToDevice, st));
    VO_TRY(vo_build_pyramids(ctx, (const uint8_t*)B->raw.p, fb, lp->cfg.batch.rows, lp->cfg.batch.cols, B->geom,
                             (uint8_t*)B->slabs[B->cur].p + (size_t)seq * sb, sb, 1, st));
    const size_t lo = (size_t)seq * d.L, co = (size_t)seq * d.C;
    if (n_lm > 0) {
        VO_CUDA(ctx, cudaMemcpyAsync(d.lm + 3 * lo, lm, (size_t)n_lm * 12, cudaMemcpyHostToDevice, st));
        VO_CUDA(ctx, cudaMemcpyAsync(d.lm_kp + 2 * lo, lm_kp, (size_t)n_lm * 8, cudaMemcpyHostToDevice, st));
    }
    if (n_cand > 0) {
        VO_CUDA(ctx, cudaMemcpyAsync(d.keys + 2 * co, keys, (size_t)n_cand * 8, cudaMemcpyHostToDevice, st));
        VO_CUDA(ctx, cudaMemcpyAsync(d.fkeys + 2 * co, first_keys, (size_t)n_cand * 8, cudaMemcpyHostToDevice, st));
        VO_CUDA(ctx, cudaMemcpyAsync(d.fpose + co, first_pose, (size_t)n_cand * 4, cudaMemcpyHostToDevice, st));
    }
    VO_CUDA(ctx, cudaMemcpyAsync(d.poses + (size_t)seq * d.P * 12, poses, (size_t)n_poses * 96, cudaMemcpyHostToDevice, st));
    const int v[6] = {n_lm, n_cand, n_poses, B200VO_LOOP_OK, n_lm, n_cand > 1 ? n_cand : 0};
    int* dst[6] = {d.n_lm, d.n_cand, d.n_poses, d.status, d.trk_lm, d.trk_cand};
    for (int i = 0; i < 6; ++i) VO_CUDA(ctx, cudaMemcpyAsync(dst[i] + seq, v + i, 4, cudaMemcpyHostToDevice, st));
    VO_CUDA(ctx, cudaStreamSynchronize(st));
    return 0;
}

extern "C" int b200vo_loop_read_state(b200vo_loop* lp, int seq, float* lm, float* lm_kp, int32_t* n_lm, float* keys, float* first_keys,
                                      int32_t* first_pose, int32_t* n_cand, double* poses, int32_t* n_poses, int32_t* status)
{
    if (!lp || !lm || !lm_kp || !n_lm || !keys || !first_keys || !first_pose || !n_cand || !poses || !n_poses || !status)
        return B200VO_E_BADARG;
    b200vo_ctx* ctx = lp->ctx;
    const LoopDev& d = lp->d;
    if (seq < 0 || seq >= lp->batch) return vo_set_err(ctx, B200VO_E_BADARG, "seq = %d is outside [0, batch = %d)", seq, lp->batch);
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int* src[4] = {d.n_lm, d.n_cand, d.n_poses, d.status};
    int32_t* dst[4] = {n_lm, n_cand, n_poses, status};
    for (int i = 0; i < 4; ++i) VO_CUDA(ctx, cudaMemcpyAsync(dst[i], src[i] + seq, 4, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaStreamSynchronize(st));
    const size_t lo = (size_t)seq * d.L, co = (size_t)seq * d.C;
    VO_CUDA(ctx, cudaMemcpyAsync(lm, d.lm + 3 * lo, (size_t)*n_lm * 12, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaMemcpyAsync(lm_kp, d.lm_kp + 2 * lo, (size_t)*n_lm * 8, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaMemcpyAsync(keys, d.keys + 2 * co, (size_t)*n_cand * 8, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaMemcpyAsync(first_keys, d.fkeys + 2 * co, (size_t)*n_cand * 8, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaMemcpyAsync(first_pose, d.fpose + co, (size_t)*n_cand * 4, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaMemcpyAsync(poses, d.poses + (size_t)seq * d.P * 12, (size_t)*n_poses * 96, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaStreamSynchronize(st));
    return 0;
}
