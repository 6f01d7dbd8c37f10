// The whole per-frame loop of the reference (VisualOdometryPipeLine.py `continuous_operation` :326-373, with the data
// flow of tests/mini_vo.py `MiniVO.step`) for a batch of independent sequences.  The VO state of every sequence --
// landmarks, candidates, pose history -- stays in device memory; one step is the batch object's tracker + pose chain
// (batch.cu), batched goodFeaturesToTrack (gftt.cu), the batched triangulation and distance filter (landmarks.cu) and
// three small kernels of this file that do what the reference does with numpy between those calls:
//   commit     stop decisions, inlier landmarks, tracked candidates, (R_CW | t_CW) from rvec | tvec
//   merge      append the triangulated landmarks, keep the too_short_baseline candidates
//   append     append the corners that pass the distance filter as candidates, append the pose
// b200vo_loop_bootstrap runs the reference's `initialization` (:209-245, :295-330) for any subset of the sequences on the device
// and writes its result straight into the state: batched SIFT (sift.cu), kNN + ratio test per sequence (knn.cu), batched
// E-RANSAC (emat.cu), batched recoverPose and triangulation (landmarks.cu) and three one-CTA-per-sequence kernels of this file:
//   boot_match     the ratio-test survivors as (pts0, pts1) pairs, in query order
//   boot_inliers   the essential-matrix inliers, in order; t * sign(t_z) of the recovered pose
//   boot_load      capacity decision, the loaded state, the current frame's pyramid, the result block
// Between steps the state lives in one canonical set of arrays; every kernel that rewrites a range reads it from a
// scratch copy (the tracker output, the compacted PnP input, the candidates after the status filter), so no kernel
// reads and writes the same slots.
#include "batch.cuh"
#include "emat.cuh"
#include "landmarks.cuh"
#include "sift.cuh"
#include "mathdev.cuh"
#include "pnp.cuh"
#include <algorithm>

#define LOOP_T 256
#define LOOP_CARRY_CTAS 32   // CTAs per sequence of the pyramid carry of a listed step

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
    // a listed step: its sequences (one CTA each, result row = CTA), nullptr: every sequence; the tracker counts of the
    // step (trk_lm / trk_cand of the listed sequences, 0 for the others)
    const int* list;
    int* step_lm; int* step_cand;
};

// The sequence of CTA `blockIdx.x` of a loop kernel: the listed sequence of that row, or the CTA's own index
__device__ __forceinline__ int loop_seq(const LoopDev& d) { return d.list ? d.list[blockIdx.x] : (int)blockIdx.x; }

// The first kernel of a listed step.  Every sequence: the tracker counts of the step (its trk_lm / trk_cand when listed, 0
// otherwise: the trackers and the pose chain do no work for it), and for one that is not listed no triangulation and no
// distance filter (tri_n and n_corner still hold its last listed step's values).  Every sequence that is not listed also
// gets its current pyramid carried from the previous frames' slab set into this step's, so that after the step set `cur`
// holds every sequence's current pyramid again.  Grid (x, batch); pos = the list row's [batch] positions.
__global__ void __launch_bounds__(256)
loop_list_kernel(LoopDev d, const int* __restrict__ pos, const uint4* __restrict__ cur_slab, uint4* __restrict__ nxt_slab,
                 size_t slab_words)
{
    const int s = blockIdx.y;
    const bool listed = pos[s] >= 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        d.step_lm[s] = listed ? d.trk_lm[s] : 0;
        d.step_cand[s] = listed ? d.trk_cand[s] : 0;
        if (!listed) { d.tri_n[s] = 0; d.n_corner[s] = 0; }
    }
    if (listed) return;
    const uint4* src = cur_slab + (size_t)s * slab_words;
    uint4* dst = nxt_slab + (size_t)s * slab_words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < slab_words; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

// Steps 3-5 of MiniVO.step and the status filter of step 2: one CTA per sequence.
__global__ void __launch_bounds__(LOOP_T)
loop_commit_kernel(LoopDev d, LoopOut out)
{
    __shared__ int s_code, s_seq;
    const int s = loop_seq(d), r = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) {
        s_seq = s;
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
        const int s = *(volatile int*)&s_seq;   // read again: a listed sequence index kept live across the call would spill
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) cw[3 * i + j] = R[3 * j + i];
        for (int i = 0; i < 3; ++i) cw[9 + i] = -R[i] * rt[3] + -R[3 + i] * rt[4] + -R[6 + i] * rt[5];
        double* hist = d.poses + ((size_t)s * d.P + d.n_poses[s]) * 12;   // appended by loop_append_kernel
        for (int k = 0; k < 12; ++k) { d.cur_pose[12 * s + k] = cw[k]; hist[k] = cw[k]; out.pose[12 * r + k] = cw[k]; }
        out.n_inl[r] = d.n_inl[s];
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
    const int nc = cta_compact<LOOP_T>(d.n_cand[s], [&](int i) { return !tracked || d.cand_status[co + i] == 1; },
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
    const int s = loop_seq(d), tid = threadIdx.x;
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
    const int nc = cta_compact<LOOP_T>(d.n_cand_b[s], [&](int i) { return !ran || d.keep[co + i] != 0; },
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
    const int s = loop_seq(d), r = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) s_st = d.status[s];
    __syncthreads();
    if (s_st == B200VO_LOOP_OK) {
        const int nc = d.n_cand[s], np = d.n_poses[s];
        const size_t co = (size_t)s * d.C, go = (size_t)s * d.G;
        const int cnt = cta_compact<LOOP_T>(d.n_corner[s], [&](int i) { return d.valid[go + i] != 0; },
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
        out.status[r] = st; out.n_lm[r] = nl; out.n_cand[r] = nc;
        if (st != B200VO_LOOP_OK) {
            out.n_inl[r] = 0;
            for (int k = 0; k < 12; ++k) out.pose[12 * r + k] = 0.0;
        }
        d.trk_lm[s] = st == B200VO_LOOP_OK ? nl : 0;
        d.trk_cand[s] = st == B200VO_LOOP_OK && nc > 1 ? nc : 0;   // the reference tracks candidates only when n > 1 (:286)
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
enum { CNT_LM, CNT_CAND, CNT_POSES, CNT_STATUS, CNT_TRK_LM, CNT_TRK_CAND, CNT_INL, CNT_CAND_B, CNT_TRI, CNT_NEW, CNT_CORNER,
       CNT_FLAGS, CNT_STEP_LM, CNT_STEP_CAND, CNT_KINDS };

struct b200vo_loop {
    b200vo_ctx* ctx = nullptr;
    b200vo_batch* B = nullptr;   // pyramids, trackers, pose chain, streams
    b200vo_loop_cfg cfg{};
    int batch = 0;
    DevBuf mem;                  // state + scratch
    DevBuf res;                  // packed result block of the host steps: pose_cw [n][12] | status | n_inliers | n_lm | n_cand
    LoopDev d{};
    TriBatchArgs tri{};
    DevBuf boot_in, boot_ws;     // b200vo_loop_bootstrap: frames and keypoint counts, everything after the matching
};

extern "C" void b200vo_loop_destroy(b200vo_loop* lp)
{
    if (!lp) return;
    cudaSetDevice(lp->ctx->device);
    cudaStreamSynchronize(lp->ctx->stream);
    for (DevBuf* b : {&lp->mem, &lp->res, &lp->boot_in, &lp->boot_ws}) if (b->p) cudaFree(b->p);
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
    if (!rc) rc = vo_reserve(ctx, lp->res, nb * 96 + 4 * nb * 4);
    if (!rc) rc = vo_reserve(ctx, B->gftt_ws, vo_gftt_batch_workspace(bc.rows, bc.cols, batch, cfg->max_corners));
    if (!rc) rc = vo_reserve(ctx, B->lists, 3 * 2 * nb * sizeof(int32_t));
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
    d.step_lm = cnt + CNT_STEP_LM * nb; d.step_cand = cnt + CNT_STEP_CAND * nb;
    d.c_obj = B->c_obj; d.c_img = B->c_img; d.c_n = B->c_n; d.inliers = B->inliers;
    TriBatchArgs& t = lp->tri;
    vo_tri_common(t.common, cfg->min_dist_landmarks, cfg->max_dist_landmarks, cfg->min_baseline_angle_deg, cfg->min_baseline_frames);
    t.intr = B->intr;
    t.cap = C; t.pose_cap = P;
    t.n = d.tri_n; t.n_poses = d.n_poses; t.cur = d.cur_pose;
    t.first_keys = d.fkeys_b; t.keys = d.keys_b; t.first_pose = d.fpose_b; t.poses = d.poses;
    t.keep = d.keep; t.lm_slot = lm_slot; t.out_lm = d.new_lm; t.out_kp = d.new_kp; t.n_new = d.n_new; t.flags = cnt + CNT_FLAGS * nb;
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

// one step of every sequence, or with n_list > 0 of the sequences list[0 .. n_list) (validated), enqueued on the ctx stream
// (the tracker and the pose chain use the batch object's streams and join it); frames_dev == nullptr: the oldest submitted
// frame set.  Result row k belongs to the k-th sequence of the step.
static int loop_core(b200vo_loop* lp, const uint8_t* frames_dev, const LoopOut& o, int n_list = 0, const int32_t* list = nullptr)
{
    b200vo_ctx* ctx = lp->ctx;
    b200vo_batch* B = lp->B;
    const b200vo_loop_cfg& c = lp->cfg;
    LoopDev& d = lp->d;
    const int nb = lp->batch;
    VO_TRY(batch_select_frames(B, frames_dev, n_list, list));
    d.list = B->step_list;
    const int n_cta = d.list ? B->step_n : nb;
    if (d.list) {
        const size_t words = B->geom.slab_bytes / 16;
        loop_list_kernel<<<dim3(LOOP_CARRY_CTAS, nb), 256, 0, ctx->stream>>>(d, d.list + nb, (const uint4*)B->slabs[B->cur].p,
                                                                             (uint4*)B->slabs[B->nxt].p, words);
        ctx->launches++;
    }
    const int* trk_lm = d.list ? d.step_lm : d.trk_lm;
    const int* trk_cand = d.list ? d.step_cand : d.trk_cand;
    VO_TRY(batch_track_pose_overlapped(B, frames_dev, d.lm_kp, d.lm, trk_lm, d.keys, trk_cand, d.lm_next, d.lm_status, d.cand_next,
                                       d.cand_status, d.pose6, d.pnp_ok, d.inl_mask, d.n_inl, nullptr));
    float* corners = nullptr;
    int* small = nullptr;
    VO_TRY(vo_gftt_batch_launch(ctx, (const uint8_t*)B->slabs[B->nxt].p + B->geom.off[0], B->geom.slab_bytes, B->geom.pitch[0],
                                c.batch.rows, c.batch.cols, nb, c.max_corners, c.quality_level, c.feature_min_dist, B->gftt_ws.p,
                                &corners, &small, B->ext, d.list, n_cta, batch_mask(B)));
    d.corners = corners; d.gftt_small = small;
    loop_commit_kernel<<<n_cta, LOOP_T, 0, ctx->stream>>>(d, o);
    ctx->launches++;
    VO_TRY(vo_triangulate_batch_launch(ctx, lp->tri, nb, ctx->stream));
    loop_merge_kernel<<<n_cta, LOOP_T, 0, ctx->stream>>>(d);
    ctx->launches++;
    VO_TRY(vo_min_distance_batch_launch(ctx, nb, d.corners, d.n_corner, d.G, d.keys, d.n_cand, d.C, (float)c.feature_min_dist, d.valid,
                                        ctx->stream));
    loop_append_kernel<<<n_cta, LOOP_T, 0, ctx->stream>>>(d, o);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    return batch_finish(B);
}

// what a full step may consume: its own frames while no set waits, or the oldest submitted set if it has no list
static int loop_check_full(b200vo_loop* lp, const uint8_t* frames)
{
    const b200vo_batch* B = lp->B;
    if (frames && B->q_count > 0)
        return vo_set_err(lp->ctx, B200VO_E_BADARG, "submitted frame sets are waiting: pass frames == NULL to consume them in order");
    if (!frames && B->q_count > 0 && !B->q_list[B->q_head].empty())
        return vo_set_err(lp->ctx, B200VO_E_BADARG, "the oldest submitted frame set lists %d sequences: consume it with the listed step",
                          (int)B->q_list[B->q_head].size());
    return 0;
}

extern "C" int b200vo_loop_step_dev(b200vo_loop* lp, const uint8_t* frames_dev, int32_t* status_dev, int32_t* n_inliers_dev,
                                    int32_t* n_lm_dev, int32_t* n_cand_dev, double* pose_cw_dev)
{
    if (!lp || !status_dev || !n_inliers_dev || !n_lm_dev || !n_cand_dev || !pose_cw_dev) return B200VO_E_BADARG;
    VO_TRY(loop_check_full(lp, frames_dev));
    VO_CUDA(lp->ctx, cudaSetDevice(lp->ctx->device));
    const LoopOut o{status_dev, n_inliers_dev, n_lm_dev, n_cand_dev, pose_cw_dev};
    return loop_core(lp, frames_dev, o);
}

// One host-buffer step of every sequence (list == nullptr) or of the n listed ones (checked): one upload of the frames,
// one read-back of the result rows, packed as pose_cw [n][12] | status | n_inliers | n_lm | n_cand
static int loop_step_host(b200vo_loop* lp, int n, const int32_t* list, const uint8_t* frames, int32_t* status, int32_t* n_inliers,
                          int32_t* n_lm, int32_t* n_cand, double* pose_cw)
{
    b200vo_ctx* ctx = lp->ctx;
    b200vo_batch* B = lp->B;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const size_t ns = n, f_total = (size_t)lp->cfg.batch.rows * lp->cfg.batch.cols * ns;
    bool pinned = false;
    if (frames) {
        cudaPointerAttributes at{};
        pinned = cudaPointerGetAttributes(&at, frames) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
    }
    uint8_t* r = (uint8_t*)lp->res.p;
    const LoopOut o{(int*)(r + ns * 96), (int*)(r + ns * 96) + ns, (int*)(r + ns * 96) + 2 * ns, (int*)(r + ns * 96) + 3 * ns, (double*)r};
    const size_t res_bytes = ns * 96 + 4 * ns * 4;
    const size_t staged = frames && !pinned ? vo_align(f_total, 256) : 0;
    VO_TRY(vo_reserve_pinned(ctx, staged + res_bytes));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    const uint8_t* fdev = nullptr;
    if (frames) {   // the one upload of the step
        VO_TRY(vo_reserve(ctx, B->raw, f_total));
        if (!pinned) memcpy(hp, frames, f_total);
        VO_CUDA(ctx, cudaMemcpyAsync(B->raw.p, pinned ? frames : hp, f_total, cudaMemcpyHostToDevice, ctx->stream));
        fdev = (const uint8_t*)B->raw.p;
    }
    VO_TRY(loop_core(lp, fdev, o, list ? n : 0, list));
    uint8_t* ho = hp + staged;   // the one read-back of the step
    VO_CUDA(ctx, cudaMemcpyAsync(ho, r, res_bytes, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    memcpy(pose_cw, ho, ns * 96);
    const int* ri = (const int*)(ho + ns * 96);
    memcpy(status, ri, ns * 4);
    memcpy(n_inliers, ri + ns, ns * 4);
    memcpy(n_lm, ri + 2 * ns, ns * 4);
    memcpy(n_cand, ri + 3 * ns, ns * 4);
    return 0;
}

extern "C" int b200vo_loop_step(b200vo_loop* lp, const uint8_t* frames, int32_t* status, int32_t* n_inliers, int32_t* n_lm,
                                int32_t* n_cand, double* pose_cw)
{
    if (!lp || !status || !n_inliers || !n_lm || !n_cand || !pose_cw) return B200VO_E_BADARG;
    VO_TRY(loop_check_full(lp, frames));
    return loop_step_host(lp, lp->batch, nullptr, frames, status, n_inliers, n_lm, n_cand, pose_cw);
}

extern "C" int b200vo_loop_submit_frames(b200vo_loop* lp, const uint8_t* frames)
{
    return lp ? batch_submit(lp->B, frames, false) : B200VO_E_BADARG;
}

extern "C" int b200vo_loop_submit_frames_dev(b200vo_loop* lp, const uint8_t* frames_dev)
{
    return lp ? batch_submit(lp->B, frames_dev, true) : B200VO_E_BADARG;
}

// ------------------------------------------------------------------------------------------
// listed steps: only the sequences of a list advance
// ------------------------------------------------------------------------------------------
// what a listed step may consume: its own frames while no set waits, or the oldest submitted set if it has the same list
static int loop_check_step_list(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames)
{
    b200vo_ctx* ctx = lp->ctx;
    const b200vo_batch* B = lp->B;
    VO_TRY(vo_check_seqs(ctx, lp->batch, n_seq, seqs));
    if (frames) {
        if (B->q_count > 0)
            return vo_set_err(ctx, B200VO_E_BADARG, "submitted frame sets are waiting: pass frames == NULL to consume them in order");
        return 0;
    }
    if (B->q_count == 0) return vo_set_err(ctx, B200VO_E_BADARG, "frames == NULL but no frame set was submitted");
    const std::vector<int32_t>& q = B->q_list[B->q_head];
    if (q.empty()) return vo_set_err(ctx, B200VO_E_BADARG, "the oldest submitted frame set covers every sequence: consume it with the full step");
    if ((int)q.size() != n_seq || !std::equal(q.begin(), q.end(), seqs))
        return vo_set_err(ctx, B200VO_E_BADARG, "the oldest submitted frame set was submitted with another list");
    return 0;
}

extern "C" int b200vo_loop_step_seqs_dev(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames_dev, int32_t* status_dev,
                                         int32_t* n_inliers_dev, int32_t* n_lm_dev, int32_t* n_cand_dev, double* pose_cw_dev)
{
    if (!lp) return B200VO_E_BADARG;
    if (!status_dev || !n_inliers_dev || !n_lm_dev || !n_cand_dev || !pose_cw_dev) return vo_set_err(lp->ctx, B200VO_E_BADARG, "null array");
    VO_TRY(loop_check_step_list(lp, n_seq, seqs, frames_dev));
    VO_CUDA(lp->ctx, cudaSetDevice(lp->ctx->device));
    const LoopOut o{status_dev, n_inliers_dev, n_lm_dev, n_cand_dev, pose_cw_dev};
    return loop_core(lp, frames_dev, o, n_seq, seqs);
}

extern "C" int b200vo_loop_step_seqs(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames, int32_t* status,
                                     int32_t* n_inliers, int32_t* n_lm, int32_t* n_cand, double* pose_cw)
{
    if (!lp) return B200VO_E_BADARG;
    if (!status || !n_inliers || !n_lm || !n_cand || !pose_cw) return vo_set_err(lp->ctx, B200VO_E_BADARG, "null array");
    VO_TRY(loop_check_step_list(lp, n_seq, seqs, frames));
    return loop_step_host(lp, n_seq, seqs, frames, status, n_inliers, n_lm, n_cand, pose_cw);
}

extern "C" int b200vo_loop_submit_frames_seqs(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames)
{
    if (!lp) return B200VO_E_BADARG;
    VO_TRY(vo_check_seqs(lp->ctx, lp->batch, n_seq, seqs));
    return batch_submit(lp->B, frames, false, n_seq, seqs);
}

extern "C" int b200vo_loop_submit_frames_seqs_dev(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames_dev)
{
    if (!lp) return B200VO_E_BADARG;
    VO_TRY(vo_check_seqs(lp->ctx, lp->batch, n_seq, seqs));
    return batch_submit(lp->B, frames_dev, true, n_seq, seqs);
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
    const int rows = lp->cfg.batch.rows, cols = lp->cfg.batch.cols;
    const size_t fb = (size_t)rows * cols;
    // the frame is tight at the sequence's own size: it becomes the top-left of a slot-layout frame
    const int rs = B->seq[seq].ext.h[0], cs = B->seq[seq].ext.w[0];
    VO_TRY(vo_reserve(ctx, B->raw, fb));
    VO_CUDA(ctx, cudaMemcpy2DAsync(B->raw.p, (size_t)cols, frame, (size_t)cs, (size_t)cs, (size_t)rs, cudaMemcpyHostToDevice, st));
    VO_TRY(batch_pyramids(B, (const uint8_t*)B->raw.p, B->cur, seq, 1, st));
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

// the listed sequences' pyramids no longer match their frames: IDLE (state arrays kept) until loaded or bootstrapped
static int loop_idle(b200vo_loop* lp, int n_seq, const int32_t* seqs)
{
    b200vo_ctx* ctx = lp->ctx;
    const int idle = B200VO_LOOP_IDLE, zero = 0;
    const LoopDev& d = lp->d;
    for (int k = 0; k < n_seq; ++k) {
        VO_CUDA(ctx, cudaMemcpyAsync(d.status + seqs[k], &idle, 4, cudaMemcpyHostToDevice, ctx->stream));
        VO_CUDA(ctx, cudaMemcpyAsync(d.trk_lm + seqs[k], &zero, 4, cudaMemcpyHostToDevice, ctx->stream));
        VO_CUDA(ctx, cudaMemcpyAsync(d.trk_cand + seqs[k], &zero, 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// The C setters: a setting that leaves the listed sequences' resident pyramids stale makes them IDLE
extern "C" int b200vo_loop_set_intrinsics(b200vo_loop* lp, int n_seq, const int32_t* seqs, const double* K)
{
    bool stale = false;
    const int rc = lp ? batch_set_intrinsics(lp->B, n_seq, seqs, K, &stale) : B200VO_E_BADARG;
    return stale ? loop_idle(lp, n_seq, seqs) : rc;
}

extern "C" int b200vo_loop_set_frame_size(b200vo_loop* lp, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols)
{
    bool stale = false;
    const int rc = lp ? batch_set_frame_size(lp->B, n_seq, seqs, rows, cols, &stale) : B200VO_E_BADARG;
    return stale ? loop_idle(lp, n_seq, seqs) : rc;
}

extern "C" int b200vo_loop_set_distortion(b200vo_loop* lp, int n_seq, const int32_t* seqs, const double* dist)
{
    bool stale = false;
    const int rc = lp ? batch_set_lens(lp->B, n_seq, seqs, nullptr, dist, nullptr, &stale) : B200VO_E_BADARG;
    return stale ? loop_idle(lp, n_seq, seqs) : rc;
}

extern "C" int b200vo_loop_set_lens(b200vo_loop* lp, int n_seq, const int32_t* seqs, const int32_t* model, const double* coeffs,
                                    const double* raw_K)
{
    bool stale = false;
    const int rc = lp ? batch_set_lens(lp->B, n_seq, seqs, model, coeffs, raw_K, &stale) : B200VO_E_BADARG;
    return stale ? loop_idle(lp, n_seq, seqs) : rc;
}

extern "C" int b200vo_loop_set_detection_mask(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* masks)
{
    bool stale = false;
    const int rc = lp ? batch_set_detection_mask(lp->B, n_seq, seqs, masks, &stale) : B200VO_E_BADARG;
    return stale ? loop_idle(lp, n_seq, seqs) : rc;
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

// ------------------------------------------------------------------------------------------
// bootstrap
// ------------------------------------------------------------------------------------------
enum { BT_SEQ, BT_QOFF, BT_NQ, BT_ROW0, BT_ROW1, BT_KINDS };   // per listed sequence, uploaded by the host

struct BootDev {
    int n_seq, cap;                            // cap: point slots per sequence (most query keypoints of any sequence)
    const int* tab;                            // [n_seq][BT_KINDS]
    const float* kp6;                          // SIFT keypoints of every frame (6 floats a row)
    const int* idx2; const uint8_t* accept;    // kNN of every sequence, rows at its query offset
    float* pts0; float* pts1; int* n_match;    // [n_seq][cap] ratio-test matches
    const uint8_t* emask; const int* eres;     // E-RANSAC inlier mask [n_seq][cap], result [n_seq][4] (found first)
    const int* eflags;                         // E-RANSAC flags [n_seq]: bit 0 = RNG table exhausted
    float* inl0; float* inl1; int* n_inl;      // the inliers: first_keys, keys
    const double* Rt;                          // recovered R | t [n_seq][12]
    double* cur; int* tri_n;                   // current pose (t * sign(t_z)) and the triangulation's point count
    const uint8_t* keep; const float* new_lm; const float* new_kp; const int* n_new;   // triangulation output
    const uint8_t* slab; size_t slab_bytes;    // pyramids of frames1 [n_seq]
    uint8_t* cur_slab;                         // the loop's current-frame slabs [batch]
    int* res;                                  // [4][n_seq] status | num_pts | n_lm | n_cand
};

// an essential matrix from cv2's sample stream (a sample draw that ran out of random numbers counts as none found)
__device__ __forceinline__ bool boot_found(const BootDev& b, int k) { return b.eres[4 * k] != 0 && !(b.eflags[k] & 1); }

__global__ void __launch_bounds__(LOOP_T)
boot_match_kernel(BootDev b)
{
    const int k = blockIdx.x;
    const int* t = b.tab + BT_KINDS * k;
    const int qo = t[BT_QOFF], nq = t[BT_NQ];
    const float* k0 = b.kp6 + (size_t)t[BT_ROW0] * 6;
    const float* k1 = b.kp6 + (size_t)t[BT_ROW1] * 6;
    const size_t po = (size_t)k * b.cap;
    const int n = cta_compact<LOOP_T>(nq, [&](int i) { return b.accept[qo + i] != 0; },
                                      [&](int i, int o) {
                                          const int j = b.idx2[2 * (qo + i)];
                                          b.pts0[2 * (po + o)] = k0[6 * i]; b.pts0[2 * (po + o) + 1] = k0[6 * i + 1];
                                          b.pts1[2 * (po + o)] = k1[6 * j]; b.pts1[2 * (po + o) + 1] = k1[6 * j + 1];
                                      });
    if (threadIdx.x == 0) b.n_match[k] = n;
}

__global__ void __launch_bounds__(LOOP_T)
boot_inliers_kernel(BootDev b)
{
    const int k = blockIdx.x;
    const bool found = boot_found(b, k);
    const size_t po = (size_t)k * b.cap;
    const int n = cta_compact<LOOP_T>(found ? b.n_match[k] : 0, [&](int i) { return b.emask[po + i] == 1; },
                                      [&](int i, int o) {
                                          b.inl0[2 * (po + o)] = b.pts0[2 * (po + i)]; b.inl0[2 * (po + o) + 1] = b.pts0[2 * (po + i) + 1];
                                          b.inl1[2 * (po + o)] = b.pts1[2 * (po + i)]; b.inl1[2 * (po + o) + 1] = b.pts1[2 * (po + i) + 1];
                                      });
    if (threadIdx.x == 0) b.n_inl[k] = n;
}

// after recoverPose: the current pose R | t * np.sign(t_z) (:317; sign(0) = 0, sign(NaN) = NaN) and the triangulation's count
__global__ void boot_pose_kernel(BootDev b)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= b.n_seq) return;
    const bool found = boot_found(b, k);
    const double* rt = b.Rt + 12 * k;
    const double tz = rt[11];
    const double sg = tz > 0 ? 1.0 : tz < 0 ? -1.0 : tz == 0 ? 0.0 : tz;
    for (int q = 0; q < 9; ++q) b.cur[12 * k + q] = rt[q];
    for (int q = 9; q < 12; ++q) b.cur[12 * k + q] = rt[q] * sg;
    b.tri_n[k] = found ? b.n_inl[k] : 0;
}

__global__ void __launch_bounds__(LOOP_T)
boot_load_kernel(LoopDev d, BootDev b)
{
    __shared__ int s_code;
    const int k = blockIdx.x, tid = threadIdx.x;
    const int s = b.tab[BT_KINDS * k + BT_SEQ];
    const size_t po = (size_t)k * b.cap;
    const bool found = boot_found(b, k);
    const int n_inl = b.n_inl[k], nn = found ? b.n_new[k] : 0;
    // the too_short_baseline candidates (keep == 1), counted before anything is written
    const int nc = cta_compact<LOOP_T>(found ? n_inl : 0, [&](int i) { return b.keep[po + i] != 0; }, [](int, int) {});
    if (tid == 0) {
        s_code = !found ? B200VO_LOOP_NO_BOOTSTRAP : (nn > d.L || nc > d.C) ? B200VO_LOOP_OVERFLOW : B200VO_LOOP_OK;
        b.res[k] = s_code;
        b.res[b.n_seq + k] = found ? n_inl : 0;
        b.res[2 * b.n_seq + k] = s_code == B200VO_LOOP_OK ? nn : 0;
        b.res[3 * b.n_seq + k] = s_code == B200VO_LOOP_OK ? nc : 0;
    }
    __syncthreads();
    if (s_code != B200VO_LOOP_OK) {   // the state arrays stay as they were; the sequence is skipped until loaded again
        if (tid == 0) { d.status[s] = s_code; d.trk_lm[s] = 0; d.trk_cand[s] = 0; }
        return;
    }
    const size_t lo = (size_t)s * d.L, co = (size_t)s * d.C;
    for (int i = tid; i < nn; i += LOOP_T) {
        d.lm[3 * (lo + i)] = b.new_lm[3 * (po + i)]; d.lm[3 * (lo + i) + 1] = b.new_lm[3 * (po + i) + 1];
        d.lm[3 * (lo + i) + 2] = b.new_lm[3 * (po + i) + 2];
        d.lm_kp[2 * (lo + i)] = b.new_kp[2 * (po + i)]; d.lm_kp[2 * (lo + i) + 1] = b.new_kp[2 * (po + i) + 1];
    }
    cta_compact<LOOP_T>(n_inl, [&](int i) { return b.keep[po + i] != 0; },
                        [&](int i, int o) {
                            d.keys[2 * (co + o)] = b.inl1[2 * (po + i)]; d.keys[2 * (co + o) + 1] = b.inl1[2 * (po + i) + 1];
                            d.fkeys[2 * (co + o)] = b.inl0[2 * (po + i)]; d.fkeys[2 * (co + o) + 1] = b.inl0[2 * (po + i) + 1];
                            d.fpose[co + o] = 0;
                        });
    double* ph = d.poses + (size_t)s * d.P * 12;   // [I | 0], [R | t]
    if (tid < 12) ph[tid] = (tid == 0 || tid == 4 || tid == 8) ? 1.0 : 0.0;
    else if (tid < 24) ph[tid] = b.cur[12 * k + tid - 12];
    const uint4* src = (const uint4*)(b.slab + (size_t)k * b.slab_bytes);
    uint4* dst = (uint4*)(b.cur_slab + (size_t)s * b.slab_bytes);
    for (size_t i = tid; i < b.slab_bytes / 16; i += LOOP_T) dst[i] = src[i];
    if (tid == 0) {
        d.n_lm[s] = nn; d.n_cand[s] = nc; d.n_poses[s] = 2; d.status[s] = B200VO_LOOP_OK;
        d.trk_lm[s] = nn; d.trk_cand[s] = nc > 1 ? nc : 0;
    }
}

extern "C" int b200vo_loop_bootstrap(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames0, const uint8_t* frames1,
                                     double ratio, int32_t* status, int32_t* num_pts, int32_t* n_lm, int32_t* n_cand)
{
    if (!lp) return B200VO_E_BADARG;
    b200vo_ctx* ctx = lp->ctx;
    b200vo_batch* B = lp->B;
    VO_TRY(vo_check_seqs(ctx, lp->batch, n_seq, seqs));
    if (!frames0 || !frames1 || !status || !num_pts || !n_lm || !n_cand) return vo_set_err(ctx, B200VO_E_BADARG, "null array");
    const int rows = lp->cfg.batch.rows, cols = lp->cfg.batch.cols;
    const size_t fb = (size_t)rows * cols, sb = B->geom.slab_bytes, ns = n_seq;
    // The sequences run in groups of one frame size (SIFT works on one size per call), the groups in the order of their
    // first listed sequence, the sequences of a group in list order: position j of the run is listed sequence perm[j].
    // Every per-sequence result depends on the sequence alone, so the order changes nothing but where it is stored.
    std::vector<int> perm, grp_end;
    {
        std::vector<char> done(ns, 0);
        for (int k = 0; k < n_seq; ++k) {
            if (done[k]) continue;
            const VoSeqExt& e = B->seq[seqs[k]].ext;
            for (int i = k; i < n_seq; ++i) {
                const VoSeqExt& f = B->seq[seqs[i]].ext;
                if (!done[i] && f.w[0] == e.w[0] && f.h[0] == e.h[0]) { done[i] = 1; perm.push_back(i); }
            }
            grp_end.push_back((int)perm.size());
        }
    }
    bool in_order = true;
    for (int j = 0; j < n_seq; ++j) in_order = in_order && perm[j] == j;
    std::vector<int32_t> seq_run(ns);
    for (int j = 0; j < n_seq; ++j) seq_run[j] = seqs[perm[j]];
    seqs = seq_run.data();
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // no step in flight reads the state
    cudaStream_t st = ctx->stream;
    // the two frames of sequence j of the run are frames 2j and 2j + 1 of the SIFT batch (slot layout)
    const size_t b_raw = vo_align(ns * 2 * fb, 256), b_cnt = vo_align(ns * 8, 256), b_moff = vo_align(ns * 16, 256);
    // sequences with distortion: the raw frames land in a staging area and are undistorted into `raw`, which then holds
    // every frame as SIFT and the second frame's pyramid read it (the pyramid build does not undistort again)
    const VoUndist ud = batch_undist(B, 0, n_seq, seqs);
    const size_t b_seq = vo_align(ns * 4, 256), b_stage = ud.xy ? b_raw + b_seq : 0;
    VO_TRY(vo_reserve(ctx, lp->boot_in, b_raw + 2 * b_cnt + b_moff + b_stage));
    uint8_t* raw = (uint8_t*)lp->boot_in.p;
    int* d_nkp = (int*)(raw + b_raw);
    int* d_row = (int*)(raw + b_raw + b_cnt);
    uint8_t* in = ud.xy ? raw + b_raw + 2 * b_cnt + b_moff : raw;   // where the raw frames land
    // both SIFT frames of a sequence with a detection mask use it: the offsets of the run's frames in the mask slab
    const VoMask mk = batch_mask(B);
    long long* d_moff = nullptr;
    if (mk.px) {
        std::vector<long long> moff(2 * ns);
        for (int j = 0; j < n_seq; ++j) moff[2 * j] = moff[2 * j + 1] = B->seq[seqs[j]].mask ? (long long)(seqs[j] * mk.stride) : -1;
        d_moff = (long long*)(raw + b_raw + 2 * b_cnt);
        VO_CUDA(ctx, cudaMemcpyAsync(d_moff, moff.data(), ns * 16, cudaMemcpyHostToDevice, st));
    }
    if (in_order) {
        VO_CUDA(ctx, cudaMemcpy2DAsync(in, 2 * fb, frames0, fb, fb, ns, cudaMemcpyHostToDevice, st));
        VO_CUDA(ctx, cudaMemcpy2DAsync(in + fb, 2 * fb, frames1, fb, fb, ns, cudaMemcpyHostToDevice, st));
    } else {
        for (int j = 0; j < n_seq; ++j) {
            VO_CUDA(ctx, cudaMemcpyAsync(in + 2 * j * fb, frames0 + (size_t)perm[j] * fb, fb, cudaMemcpyHostToDevice, st));
            VO_CUDA(ctx, cudaMemcpyAsync(in + (2 * j + 1) * fb, frames1 + (size_t)perm[j] * fb, fb, cudaMemcpyHostToDevice, st));
        }
    }
    if (ud.xy) {   // frames 2j and 2j + 1 are sequence seqs[j]'s (run order)
        int* d_seq = (int*)(in + b_raw);
        VO_CUDA(ctx, cudaMemcpyAsync(d_seq, seqs, ns * 4, cudaMemcpyHostToDevice, st));
        VO_TRY(vo_undistort_frames(ctx, in, raw, fb, (size_t)cols, 2 * n_seq, rows, cols, ud, d_seq, 1, B->ext, st));
    }
    // SIFT per size group, each group's keypoint and descriptor rows after the previous group's
    int n_rows = 0;
    for (size_t g = 0, j0 = 0; g < grp_end.size(); j0 = grp_end[g++]) {
        const VoSeqExt& e = B->seq[seqs[j0]].ext;
        const int m = grp_end[g] - (int)j0;
        VO_TRY(vo_sift_frames(ctx, raw + 2 * j0 * fb, fb, 2 * m, e.h[0], e.w[0], true, d_nkp + 2 * j0, d_row + 2 * j0, &n_rows, n_rows,
                              (size_t)cols, mk.px, d_moff ? d_moff + 2 * j0 : nullptr));
    }
    std::vector<int> h_cnt(4 * ns);
    VO_CUDA(ctx, cudaMemcpyAsync(h_cnt.data(), d_nkp, ns * 8, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaMemcpyAsync(h_cnt.data() + 2 * ns, d_row, ns * 8, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaStreamSynchronize(st));
    // per sequence: its query rows, and no matching where knnMatch has no pair to offer (no query descriptors) or the ratio
    // test cannot run (fewer than two train descriptors)
    std::vector<int> tab(BT_KINDS * ns);
    int sum_q = 0, cap = 1;
    for (int k = 0; k < n_seq; ++k) {
        const int nq = h_cnt[2 * k], nt = h_cnt[2 * k + 1];
        int* t = tab.data() + BT_KINDS * k;
        t[BT_SEQ] = seqs[k]; t[BT_QOFF] = sum_q; t[BT_NQ] = nq > 0 && nt >= 2 ? nq : 0;
        t[BT_ROW0] = h_cnt[2 * ns + 2 * k]; t[BT_ROW1] = h_cnt[2 * ns + 2 * k + 1];
        sum_q += t[BT_NQ];
        cap = std::max(cap, t[BT_NQ]);
    }
    const size_t nc = ns * cap, sq = std::max(sum_q, 1);
    const size_t sizes[] = {ns * BT_KINDS * 4, sq * 8, sq * 8, sq, nc * 8, nc * 8, ns * 4, ns * 72, nc, ns * 16, ns * 4,
                            nc * 8, nc * 8, ns * 4, nc * 4, ns * 384, ns * 16, ns * 96, ns * 8, ns * 96, ns * 4, ns * 4, ns * 96,
                            nc, nc * 12, nc * 12, nc * 8, ns * 4, ns * 4, ns * 16, ns * sb, ns * sizeof(VoSeqExt), ns * sizeof(VoIntrinsics)};
    size_t total = 0;
    for (size_t x : sizes) total += vo_align(x, 256);
    VO_TRY(vo_reserve(ctx, lp->boot_ws, total));
    uint8_t* p = (uint8_t*)lp->boot_ws.p;
    int q = 0;
    auto take = [&]() { uint8_t* r = p; p += vo_align(sizes[q++], 256); return (void*)r; };
    BootDev b{};
    b.n_seq = n_seq; b.cap = cap;
    int* d_tab = (int*)take();
    int* idx2 = (int*)take(); float* dist2 = (float*)take(); uint8_t* accept = (uint8_t*)take();
    b.tab = d_tab; b.idx2 = idx2; b.accept = accept;
    b.kp6 = (const float*)ctx->d_sift_out[0].p;
    b.pts0 = (float*)take(); b.pts1 = (float*)take(); b.n_match = (int*)take();
    double* E = (double*)take(); uint8_t* emask = (uint8_t*)take(); int* eres = (int*)take(); int* eflags = (int*)take();
    b.emask = emask; b.eres = eres; b.eflags = eflags;
    b.inl0 = (float*)take(); b.inl1 = (float*)take(); b.n_inl = (int*)take();
    int* zeros = (int*)take();
    RecArgs ra{};
    ra.poses = (double*)take(); ra.good = (int*)take(); ra.Rt = (double*)take(); ra.win = (int*)take();
    b.Rt = ra.Rt;
    b.cur = (double*)take(); b.tri_n = (int*)take();
    int* one = (int*)take();
    double* first_pose_cw = (double*)take();
    TriBatchArgs t = lp->tri;
    t.cap = cap; t.pose_cap = 1;
    t.keep = (uint8_t*)take(); t.lm_slot = (float*)take(); t.out_lm = (float*)take(); t.out_kp = (float*)take();
    t.n_new = (int*)take(); t.flags = (int*)take();
    b.res = (int*)take();
    uint8_t* slab = (uint8_t*)take();
    VoSeqExt* ext_run = (VoSeqExt*)take();
    // the camera of each listed sequence, in list order (the bootstrap's kernels take the sequence from the grid)
    VoIntrinsics* intr = (VoIntrinsics*)take();
    std::vector<VoIntrinsics> h_intr(ns);
    for (int k = 0; k < n_seq; ++k) h_intr[k] = B->seq[seqs[k]].intr;
    VO_CUDA(ctx, cudaMemcpyAsync(intr, h_intr.data(), ns * sizeof(VoIntrinsics), cudaMemcpyHostToDevice, st));
    t.intr = intr;
    b.keep = t.keep; b.new_lm = t.out_lm; b.new_kp = t.out_kp; b.n_new = t.n_new;
    b.slab = slab; b.slab_bytes = sb; b.cur_slab = (uint8_t*)B->slabs[B->cur].p;
    VO_CUDA(ctx, cudaMemcpyAsync(d_tab, tab.data(), ns * BT_KINDS * 4, cudaMemcpyHostToDevice, st));
    // the triangulation's pose history [I | 0] and every first_pose 0 (:310-313)
    std::vector<double> id(ns * 12, 0.0);
    std::vector<int> ones(ns, 1);
    for (size_t k = 0; k < ns; ++k) id[12 * k] = id[12 * k + 4] = id[12 * k + 8] = 1.0;
    VO_CUDA(ctx, cudaMemcpyAsync(first_pose_cw, id.data(), ns * 96, cudaMemcpyHostToDevice, st));
    VO_CUDA(ctx, cudaMemcpyAsync(one, ones.data(), ns * 4, cudaMemcpyHostToDevice, st));
    VO_CUDA(ctx, cudaMemsetAsync(zeros, 0, nc * 4, st));
    VO_CUDA(ctx, cudaMemsetAsync(t.flags, 0, ns * 4, st));
    // kNN(k=2) + ratio test per sequence (query: frame 0, train: frame 1), back to back on the ctx stream, in a workspace
    // reserved once for the largest of them
    size_t knn_ws = 0;
    for (int k = 0; k < n_seq; ++k)
        if (tab[BT_KINDS * k + BT_NQ] > 0) knn_ws = std::max(knn_ws, vo_knn2_workspace(ctx, tab[BT_KINDS * k + BT_NQ], h_cnt[2 * k + 1]));
    VO_TRY(vo_reserve(ctx, ctx->d_scratch[3], knn_ws));
    const float* desc = (const float*)ctx->d_sift_out[1].p;
    for (int k = 0; k < n_seq; ++k) {
        const int* tk = tab.data() + BT_KINDS * k;
        if (tk[BT_NQ] == 0) continue;
        VO_TRY(vo_knn2_ratio_dev(ctx, desc + (size_t)tk[BT_ROW0] * 128, tk[BT_NQ], desc + (size_t)tk[BT_ROW1] * 128, h_cnt[2 * k + 1], ratio,
                                 idx2 + 2 * tk[BT_QOFF], dist2 + 2 * tk[BT_QOFF], accept + tk[BT_QOFF], nullptr));
    }
    boot_match_kernel<<<n_seq, LOOP_T, 0, st>>>(b);
    ctx->launches++;
    // findEssentialMat(RANSAC, prob 0.99, threshold 1.0 = VO_BOOT_EMAT_THR, maxIters 1000) at :308
    VO_TRY(vo_emat_batch(ctx, b.pts0, b.pts1, cap, b.n_match, cap, n_seq, intr, 0.99, 1000, E, emask, eres, eflags));
    boot_inliers_kernel<<<n_seq, LOOP_T, 0, st>>>(b);
    ctx->launches++;
    // recoverPose(E, inliers, K) with distanceThresh 50 (:315)
    ra.E = E; ra.valid = eres; ra.valid_stride = 4;
    ra.intr = intr; ra.dist = 50.0;
    ra.cap = cap; ra.n = b.n_inl; ra.p1 = b.inl0; ra.p2 = b.inl1;
    VO_TRY(vo_recover_pose_batch_launch(ctx, ra, n_seq, cap, st));
    boot_pose_kernel<<<(n_seq + 127) / 128, 128, 0, st>>>(b);
    ctx->launches++;
    t.n = b.tri_n; t.n_poses = one; t.cur = b.cur;
    t.first_keys = b.inl0; t.keys = b.inl1; t.first_pose = zeros; t.poses = first_pose_cw;
    VO_TRY(vo_triangulate_batch_launch(ctx, t, n_seq, st));
    // the second frames' pyramids, each at its sequence's size (the run's own table; none while every size is the slot's)
    std::vector<VoSeqExt> h_ext(ns);
    for (int j = 0; j < n_seq; ++j) h_ext[j] = B->seq[seqs[j]].ext;
    if (B->ext) VO_CUDA(ctx, cudaMemcpyAsync(ext_run, h_ext.data(), ns * sizeof(VoSeqExt), cudaMemcpyHostToDevice, st));
    VO_TRY(vo_build_pyramids(ctx, raw + fb, 2 * fb, rows, cols, B->geom, slab, sb, n_seq, st, B->ext ? ext_run : nullptr,
                             B->ext ? h_ext.data() : nullptr));
    boot_load_kernel<<<n_seq, LOOP_T, 0, st>>>(lp->d, b);
    ctx->launches++;
    VO_CUDA(ctx, cudaGetLastError());
    std::vector<int> h_res(4 * ns);
    VO_CUDA(ctx, cudaMemcpyAsync(h_res.data(), b.res, ns * 16, cudaMemcpyDeviceToHost, st));
    VO_CUDA(ctx, cudaStreamSynchronize(st));
    for (int j = 0; j < n_seq; ++j) {   // back to list order
        const int k = perm[j];
        status[k] = h_res[j]; num_pts[k] = h_res[ns + j]; n_lm[k] = h_res[2 * ns + j]; n_cand[k] = h_res[3 * ns + j];
    }
    return 0;
}
