// Batched per-frame hot path for independent sequences (BASELINE config 5): per sequence and
// frame the reference runs calcOpticalFlowPyrLK on the landmark keypoints and on the candidate
// keypoints (VisualOdometryPipeLine.py:281,:287), keeps status==1 (:282-284), then
// solvePnPRansac on the surviving landmarks (:343).  Here one launch of each kernel covers every
// sequence of the batch, the previous frame's pyramid stays resident in HBM between steps, and
// nothing returns to the host between KLT and PnP.
#include "batch.cuh"
#include <chrono>
#include "pnp.cuh"

static void prof_mark(b200vo_batch* B, int stage, cudaStream_t stream)
{
    if (!B->profile || B->prof_n >= B200VO_PROF_RING) return;
    cudaEventRecord(B->prof_ev[B->prof_n][stage], stream);
}

// status==1 landmarks, in order, into the compact PnP input arrays (what `matched_pts[tracked]`
// does in the reference, :282-284)
__global__ void __launch_bounds__(256)
compact_tracked_kernel(int cap, const int* __restrict__ n_lm, const float* __restrict__ lm_next,
                       const uint8_t* __restrict__ lm_status, const float* __restrict__ lm_obj,
                       float* __restrict__ c_obj, float* __restrict__ c_img, int* __restrict__ c_n,
                       int* __restrict__ c_orig)
{
    const int b = blockIdx.x;
    const int n = min(max(n_lm[b], 0), cap);   // a count beyond the slot capacity must not reach the neighbour's arrays
    const size_t sb = (size_t)b * cap;
    const int cnt = cta_compact<256>(n, [&](int i) { return lm_status[sb + i] == 1; },
                                     [&](int i, int k) {
                                         const size_t gi = sb + i, o = sb + k;
                                         c_obj[3 * o] = lm_obj[3 * gi]; c_obj[3 * o + 1] = lm_obj[3 * gi + 1]; c_obj[3 * o + 2] = lm_obj[3 * gi + 2];
                                         c_img[2 * o] = lm_next[2 * gi]; c_img[2 * o + 1] = lm_next[2 * gi + 1];
                                         c_orig[o] = i;
                                     });
    if (threadIdx.x == 0) c_n[b] = cnt;
}

// inlier mask over the ORIGINAL landmark slots
__global__ void __launch_bounds__(256)
scatter_mask_kernel(int cap, const uint8_t* __restrict__ ok, const int* __restrict__ n_inl,
                    const int* __restrict__ inliers, const int* __restrict__ c_orig,
                    uint8_t* __restrict__ mask_out, int* __restrict__ n_inl_out, uint8_t* __restrict__ ok_out)
{
    const int b = blockIdx.x;
    for (int i = threadIdx.x; i < cap; i += blockDim.x) mask_out[(size_t)b * cap + i] = 0;
    __syncthreads();
    const int m = ok[b] ? n_inl[b] : 0;
    for (int k = threadIdx.x; k < m; k += blockDim.x)
        mask_out[(size_t)b * cap + c_orig[(size_t)b * cap + inliers[(size_t)b * cap + k]]] = 1;
    if (threadIdx.x == 0) { n_inl_out[b] = m; ok_out[b] = ok[b]; }
}

extern "C" int b200vo_batch_create(b200vo_ctx* ctx, int batch, const b200vo_batch_cfg* cfg, b200vo_batch** out)
{
    if (!ctx || !cfg || !out || batch <= 0) return B200VO_E_BADARG;
    *out = nullptr;
    if (cfg->max_level < 0 || cfg->win_w <= 2 || cfg->win_h <= 2 || cfg->rows <= 0 || cfg->cols <= 0)
        return vo_set_err(ctx, B200VO_E_BADARG, "maxLevel >= 0 && winSize.width > 2 && winSize.height > 2");
    if (cfg->win_w >= VO_BORDER || cfg->win_h >= VO_BORDER || cfg->cols <= cfg->win_w || cfg->rows <= cfg->win_h)
        return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "unsupported window / image size");
    if (cfg->max_landmarks < 4 || cfg->max_candidates < 0 || cfg->pnp_iters < 1)
        return vo_set_err(ctx, B200VO_E_BADARG, "bad capacities");
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    b200vo_batch* B = new b200vo_batch();
    B->ctx = ctx; B->batch = batch; B->cfg = *cfg; B->cur = 0; B->primed = false;
    const int levels = vo_pyr_levels(cfg->cols, cfg->rows, cfg->win_w, cfg->win_h, cfg->max_level);
    vo_pyr_geom(cfg->rows, cfg->cols, levels, &B->geom);
    B->kp.win_w = cfg->win_w; B->kp.win_h = cfg->win_h;
    B->kp.max_count = (cfg->crit_type & 1) ? (cfg->crit_max_count < 0 ? 0 : cfg->crit_max_count > 100 ? 100 : cfg->crit_max_count) : 30;
    double eps = (cfg->crit_type & 2) ? (cfg->crit_eps < 0 ? 0 : cfg->crit_eps > 10 ? 10 : cfg->crit_eps) : 0.01;
    B->kp.eps_sq = eps * eps;
    B->kp.min_eig_thr = (float)cfg->min_eig_thr;
    int rc = 0;
    for (int s = 0; s < 3 && !rc; ++s) rc = vo_reserve(ctx, B->slabs[s], B->geom.slab_bytes * batch);
    const int cap = cfg->max_landmarks;
    const size_t b_obj = vo_align((size_t)batch * cap * 12, 256), b_img = vo_align((size_t)batch * cap * 8, 256);
    const size_t b_n = vo_align((size_t)batch * 4, 256), b_i = vo_align((size_t)batch * cap * 4, 256);
    const size_t b_m = vo_align((size_t)batch * cap, 256);
    const size_t b_ws = vo_pnp_workspace_bytes(batch, cap, cfg->pnp_iters);
    if (!rc) rc = vo_reserve(ctx, B->work, b_obj + b_img + b_n + 2 * b_i + b_m + b_ws);
    B->n_raw = 8 * cfg->pnp_iters + 256;
    if (!rc) rc = vo_rng_table(ctx, B->n_raw, &B->rng);
    if (rc) { b200vo_batch_destroy(B); return rc; }
    {   // streams and events: any failure (descriptor / memory exhaustion with many batches) unwinds the whole object
        cudaError_t ce = cudaSuccess;
        auto ok = [&](cudaError_t e) { if (ce == cudaSuccess) ce = e; };
        int least = 0, greatest = 0;
        ok(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        ok(cudaStreamCreateWithFlags(&B->pre_stream, cudaStreamNonBlocking));
        // chunk streams carry pyramids + the landmark tracker: ahead of the candidate tracker on the ctx stream
        for (auto& st : B->chunk_stream) ok(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, greatest));
        for (auto& e : B->chunk_ev) ok(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : B->copy_ev) ok(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ok(cudaEventCreateWithFlags(&B->done_ev, cudaEventDisableTiming));
        ok(cudaStreamCreateWithFlags(&B->io_stream, cudaStreamNonBlocking));
        for (cudaEvent_t* e : {&B->obj_ev, &B->klt_ev, &B->io_ev, &B->lm_ev, &B->cand_ev, &B->pose_ev, &B->cand_in_ev})
            ok(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        ok(cudaStreamCreateWithPriority(&B->pose_stream, cudaStreamNonBlocking, greatest));
        for (auto& e : B->q_ev) ok(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ok(cudaEventCreateWithFlags(&B->step_end_ev, cudaEventDisableTiming));
        if (ce != cudaSuccess) {
            b200vo_batch_destroy(B);
            return vo_cuda_fail(ctx, ce, "b200vo_batch_create: stream / event creation");
        }
    }
    uint8_t* p = (uint8_t*)B->work.p;
    B->c_obj = (float*)p; p += b_obj;
    B->c_img = (float*)p; p += b_img;
    B->c_n = (int*)p; p += b_n;
    B->c_orig = (int*)p; p += b_i;
    B->inliers = (int*)p; p += b_i;
    B->c_mask = p; p += b_m;
    B->pnp_ws = p;
    // every sequence starts with cfg->K
    B->intr_host.resize(batch);
    vo_intrinsics_row(B->intr_host[0], cfg->K, VO_BOOT_EMAT_THR);
    for (int k = 1; k < batch; ++k) B->intr_host[k] = B->intr_host[0];
    rc = vo_reserve(ctx, B->intr_buf, (size_t)batch * sizeof(VoIntrinsics));
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(B->intr_buf.p, B->intr_host.data(), (size_t)batch * sizeof(VoIntrinsics), cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = vo_cuda_fail(ctx, e, "b200vo_batch_create: intrinsics upload");
    }
    if (rc) { b200vo_batch_destroy(B); return rc; }
    B->intr = (const VoIntrinsics*)B->intr_buf.p;
    // every sequence starts with the slot size (no table on the device until a sequence is given another)
    B->ext_host.resize(batch);
    vo_seq_ext(cfg->rows, cfg->cols, cfg->win_w, cfg->win_h, cfg->max_level, &B->ext_host[0]);
    for (int k = 1; k < batch; ++k) B->ext_host[k] = B->ext_host[0];
    rc = vo_reserve(ctx, B->ext_buf, (size_t)batch * sizeof(VoSeqExt));
    if (rc) { b200vo_batch_destroy(B); return rc; }
    *out = B;
    return 0;
}

int batch_set_intrinsics(b200vo_batch* B, int n_seq, const int32_t* seqs, const double* K)
{
    b200vo_ctx* ctx = B->ctx;
    std::vector<VoIntrinsics> rows = B->intr_host;
    VO_TRY(vo_intrinsics_set(ctx, B->batch, n_seq, seqs, K, VO_BOOT_EMAT_THR, rows.data()));
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // no step in flight reads the rows (every stream of a step joins the ctx stream)
    VO_CUDA(ctx, cudaMemcpyAsync(B->intr_buf.p, rows.data(), rows.size() * sizeof(VoIntrinsics), cudaMemcpyHostToDevice, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B->intr_host.swap(rows);
    return 0;
}

extern "C" int b200vo_batch_set_intrinsics(b200vo_batch* B, int n_seq, const int32_t* seqs, const double* K)
{
    return B ? batch_set_intrinsics(B, n_seq, seqs, K) : B200VO_E_BADARG;
}

int batch_set_frame_size(b200vo_batch* B, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols)
{
    b200vo_ctx* ctx = B->ctx;
    const b200vo_batch_cfg& c = B->cfg;
    if (n_seq < 1 || n_seq > B->batch) return vo_set_err(ctx, B200VO_E_BADARG, "n_seq = %d is outside [1, batch = %d]", n_seq, B->batch);
    if (!seqs || !rows || !cols) return vo_set_err(ctx, B200VO_E_BADARG, "null array");
    std::vector<char> seen(B->batch, 0);
    for (int k = 0; k < n_seq; ++k) {
        if (seqs[k] < 0 || seqs[k] >= B->batch)
            return vo_set_err(ctx, B200VO_E_BADARG, "seqs[%d] = %d is outside [0, batch = %d)", k, seqs[k], B->batch);
        if (seen[seqs[k]]++) return vo_set_err(ctx, B200VO_E_BADARG, "sequence %d is listed twice", seqs[k]);
        // the slot bounds the frame; the window bounds it from below as it bounds cfg->rows / cfg->cols (and with it the
        // detector's 3 x 3 minimum)
        if (rows[k] > c.rows || cols[k] > c.cols)
            return vo_set_err(ctx, B200VO_E_BADARG, "sequence %d: %d x %d does not fit the %d x %d slot", seqs[k], rows[k], cols[k], c.rows, c.cols);
        if (rows[k] <= c.win_h || cols[k] <= c.win_w)
            return vo_set_err(ctx, B200VO_E_BADARG, "sequence %d: %d x %d is not larger than the %d x %d window", seqs[k], rows[k], cols[k],
                              c.win_h, c.win_w);
    }
    if (B->q_count > 0) return vo_set_err(ctx, B200VO_E_BADARG, "submitted frame sets are waiting: their pyramids were built at the old sizes");
    std::vector<VoSeqExt> ext = B->ext_host;
    for (int k = 0; k < n_seq; ++k) vo_seq_ext(rows[k], cols[k], c.win_w, c.win_h, c.max_level, &ext[seqs[k]]);
    bool uniform = true;
    for (const VoSeqExt& e : ext) uniform = uniform && e.w[0] == c.cols && e.h[0] == c.rows;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // no step in flight reads the rows
    VO_CUDA(ctx, cudaStreamSynchronize(B->pre_stream));
    VO_CUDA(ctx, cudaMemcpyAsync(B->ext_buf.p, ext.data(), ext.size() * sizeof(VoSeqExt), cudaMemcpyHostToDevice, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B->ext_host.swap(ext);
    B->ext = uniform ? nullptr : (const VoSeqExt*)B->ext_buf.p;
    return 0;
}

extern "C" int b200vo_batch_set_frame_size(b200vo_batch* B, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols)
{
    if (!B) return B200VO_E_BADARG;
    VO_TRY(batch_set_frame_size(B, n_seq, seqs, rows, cols));
    B->primed = false;   // the resident pyramids were built at the old sizes
    return 0;
}

__global__ void trace_stamp_kernel(unsigned long long* dst)
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    *dst = t;
}

// B200VO_TRACE_FILE=<path>: when the batch is destroyed, write where and when (GPU wall clock, ns) the pose CTAs of the LAST
// step ran and when the most recent tracker launches claimed their first feature / retired their last warp -- the
// picture of how the pose chain and the candidate tracker share the machine that CUDA events cannot give.
static void batch_write_trace(b200vo_batch* B)
{
    const char* path = getenv("B200VO_TRACE_FILE");
    if (!path || !B->trace.p) return;
    cudaDeviceSynchronize();
    std::vector<long long> t((size_t)B->batch * 16);
    if (cudaMemcpy(t.data(), B->trace.p, t.size() * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return;
    std::vector<unsigned long long> q;
    vo_klt_trace_read(B->ctx, q);
    FILE* f = fopen(path, "w");
    if (!f) return;
    long long t0 = 0;
    for (int b = 0; b < B->batch; ++b) if (!t0 || (t[(size_t)b * 16 + 12] && t[(size_t)b * 16 + 12] < t0)) t0 = t[(size_t)b * 16 + 12];
    fprintf(f, "# pose CTAs of the last step: sequence, SM, start and end in us after the first pose CTA started\n");
    for (int b = 0; b < B->batch; ++b)
        fprintf(f, "pose %d sm %lld start %.1f end %.1f\n", b, t[(size_t)b * 16 + 13], (t[(size_t)b * 16 + 12] - t0) * 1e-3,
                (t[(size_t)b * 16 + 14] - t0) * 1e-3);
    if (B->host_n)
        fprintf(f, "# host side of b200vo_batch_step, mean us over %ld calls: inputs enqueued %.1f, kernels enqueued %.1f, read-back enqueued %.1f, "
                   "synchronised %.1f, returned %.1f; between calls %.1f\n", B->host_n, B->host_us[0] / B->host_n, B->host_us[1] / B->host_n,
                B->host_us[2] / B->host_n, B->host_us[3] / B->host_n, B->host_us[4] / B->host_n, B->host_us[5] / B->host_n);
    if (B->stamps.p) {
        std::vector<unsigned long long> st(64 * 4);
        if (cudaMemcpy(st.data(), B->stamps.p, st.size() * 8, cudaMemcpyDeviceToHost) == cudaSuccess) {
            fprintf(f, "# host-buffer steps, same clock: point arrays uploaded (first kernel may start), results read back (the call returns)\n");
            for (long k = B->stamp_step > 24 ? B->stamp_step - 24 : 0; k < B->stamp_step; ++k)
                fprintf(f, "step %ld uploaded %.1f read_back %.1f (candidate results: from %.1f to %.1f)\n", k, ((long long)st[(k & 63) * 4] - t0) * 1e-3,
                        ((long long)st[(k & 63) * 4 + 1] - t0) * 1e-3, ((long long)st[(k & 63) * 4 + 2] - t0) * 1e-3, ((long long)st[(k & 63) * 4 + 3] - t0) * 1e-3);
        }
    }
    fprintf(f, "# tracker launches (queue ring), same clock: first feature claimed, last warp retired\n");
    for (size_t i = 0; i + 1 < q.size(); i += 2)
        if (q[i] && (long long)q[i + 1] > t0 - 60000000)
            fprintf(f, "klt slot %d start %.1f end %.1f\n", (int)(i / 2), ((long long)q[i] - t0) * 1e-3, ((long long)q[i + 1] - t0) * 1e-3);
    fclose(f);
}

extern "C" void b200vo_batch_destroy(b200vo_batch* B)
{
    if (!B) return;
    cudaSetDevice(B->ctx->device);
    cudaStreamSynchronize(B->ctx->stream);
    batch_write_trace(B);
    if (B->trace.p) cudaFree(B->trace.p);
    if (B->stamps.p) cudaFree(B->stamps.p);
    auto kill_stream = [](cudaStream_t st) { if (st) { cudaStreamSynchronize(st); cudaStreamDestroy(st); } };
    auto kill_event = [](cudaEvent_t e) { if (e) cudaEventDestroy(e); };
    kill_stream(B->pre_stream);
    for (auto& st : B->chunk_stream) kill_stream(st);
    kill_stream(B->io_stream);
    kill_stream(B->pose_stream);
    for (auto& s : B->slabs) if (s.p) cudaFree(s.p);
    for (DevBuf* d : {&B->raw, &B->raw_pre, &B->pts_in, &B->outs, &B->work, &B->gftt_ws, &B->intr_buf, &B->ext_buf, &B->lists})
        if (d->p) cudaFree(d->p);
    for (auto& e : B->q_ev) kill_event(e);
    for (auto& e : B->chunk_ev) kill_event(e);
    for (auto& e : B->copy_ev) kill_event(e);
    for (cudaEvent_t e : {B->step_end_ev, B->done_ev, B->obj_ev, B->klt_ev, B->io_ev, B->lm_ev, B->cand_ev, B->pose_ev, B->cand_in_ev}) kill_event(e);
    if (B->prof_init) for (auto& row : B->prof_ev) for (auto& e : row) kill_event(e);
    cudaGetLastError();
    delete B;
}

static int batch_upload_frames(b200vo_batch* B, const uint8_t* frames, int slab_set)
{
    b200vo_ctx* ctx = B->ctx;
    const size_t fb = (size_t)B->cfg.rows * B->cfg.cols;
    const size_t total = fb * B->batch;
    VO_TRY(vo_reserve(ctx, B->raw, total));
    cudaPointerAttributes at{};
    const bool pinned = cudaPointerGetAttributes(&at, frames) == cudaSuccess && at.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const uint8_t* src = frames;
    if (!pinned) {   // pageable caller memory: stage through the ctx's pinned buffer
        VO_TRY(vo_reserve_pinned(ctx, total));
        memcpy(ctx->h_pin, frames, total);
        src = (const uint8_t*)ctx->h_pin;
    }
    VO_CUDA(ctx, cudaMemcpyAsync(B->raw.p, src, total, cudaMemcpyHostToDevice, ctx->stream));
    VO_TRY(vo_build_pyramids(ctx, (const uint8_t*)B->raw.p, fb, B->cfg.rows, B->cfg.cols, B->geom,
                             (uint8_t*)B->slabs[slab_set].p, B->geom.slab_bytes, B->batch, ctx->stream, batch_ext_dev(B, 0), batch_ext_host(B, 0)));
    return 0;
}

// a slab set that neither holds the previous frames nor a prefetched frame set
int batch_free_set(const b200vo_batch* B)
{
    for (int s = 0; s < 3; ++s) {
        bool used = s == B->cur;
        for (int k = 0; k < B->q_count; ++k) used = used || B->q_set[(B->q_head + k) & 1] == s;
        if (!used) return s;
    }
    return -1;
}

// the device row of a list: [list | pos], see b200vo_batch::lists
static int* batch_list_row(const b200vo_batch* B, int row) { return (int*)B->lists.p + (size_t)row * 2 * B->batch; }

// upload a list into its device row on `stream` (a pageable source: staged before the call returns, nothing waits)
static int batch_upload_list(b200vo_batch* B, int row, int n, const int32_t* list, cudaStream_t stream)
{
    std::vector<int32_t> r(2 * (size_t)B->batch, -1);
    for (int k = 0; k < n; ++k) { r[k] = list[k]; r[B->batch + list[k]] = k; }
    VO_CUDA(B->ctx, cudaMemcpyAsync(batch_list_row(B, row), r.data(), r.size() * 4, cudaMemcpyHostToDevice, stream));
    return 0;
}

// Frames of a FUTURE step: copied and turned into pyramids on a side stream while the current step's
// kernels run; the step that passes frames == NULL consumes them (oldest first).
int batch_submit(b200vo_batch* B, const uint8_t* frames, bool dev, int n_list, const int32_t* list)
{
    if (!B || !frames) return B200VO_E_BADARG;
    b200vo_ctx* ctx = B->ctx;
    if (!B->primed) return vo_set_err(ctx, B200VO_E_BADARG, "b200vo_batch_prime was not called");
    if (B->q_count >= 2) return vo_set_err(ctx, B200VO_E_BADARG, "two frame sets are already waiting for their step");
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    const int set = batch_free_set(B);
    if (set < 0) return vo_set_err(ctx, B200VO_E_BADARG, "no free pyramid set");
    const size_t fb = (size_t)B->cfg.rows * B->cfg.cols, total = fb * B->batch;
    cudaPointerAttributes at{};
    const bool known = cudaPointerGetAttributes(&at, frames) == cudaSuccess;
    cudaGetLastError();
    if (dev) {
        if (!known || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged))
            return vo_set_err(ctx, B200VO_E_BADARG, "b200vo_batch_submit_frames_dev needs a device pointer");
    } else {
        VO_TRY(vo_reserve(ctx, B->raw_pre, total));
        if (!known || at.type != cudaMemoryTypeHost)
            return vo_set_err(ctx, B200VO_E_BADARG, "submitted frames must live in page-locked memory (b200vo_host_alloc)");
    }
    const int slot = (B->q_head + B->q_count) & 1;
    B->q_set[slot] = set;
    B->q_src[slot] = frames;
    B->q_dev[slot] = dev;
    B->q_list[slot].assign(list, list + n_list);
    B->q_count++;
    return 0;
}

extern "C" int b200vo_batch_submit_frames(b200vo_batch* B, const uint8_t* frames) { return batch_submit(B, frames, false); }

// The same for frames that are already resident (and complete) in device memory: no copy, the pyramids are built from
// the caller's buffer on the side stream while the step in flight runs; b200vo_batch_step_dev(frames_dev == NULL)
// consumes them.  The buffer must stay untouched until that step has been enqueued.
extern "C" int b200vo_batch_submit_frames_dev(b200vo_batch* B, const uint8_t* frames_dev) { return batch_submit(B, frames_dev, true); }

// Enqueue the copies + pyramid builds of the submitted frame sets that are still waiting.  Called
// from inside the next step and ordered (event `after`) behind that step's own small uploads: the
// copy engine arbitrates between streams per copy, not in enqueue order, and a 30 MB frame copy
// slipping in between the point arrays holds the step's first kernel back by the whole copy
// (measured: 0.6 ms instead of 0.06 ms for the uploads).
int batch_issue_prefetch(b200vo_batch* B, cudaEvent_t after, bool wait_step_end)
{
    b200vo_ctx* ctx = B->ctx;
    const size_t fb = (size_t)B->cfg.rows * B->cfg.cols, total = fb * B->batch;
    for (int k = 0; k < B->q_count; ++k) {
        const int slot = (B->q_head + k) & 1;
        if (!B->q_src[slot]) continue;
        if (wait_step_end) VO_CUDA(ctx, cudaStreamWaitEvent(B->pre_stream, B->step_end_ev, 0));   // readers of this set have retired
        if (after) VO_CUDA(ctx, cudaStreamWaitEvent(B->pre_stream, after, 0));  // and the step's own uploads have landed
        const std::vector<int32_t>& ql = B->q_list[slot];
        // a listed set: its list row was last read by the step that consumed the slot's previous set, which ended before
        // step_end_ev (the pyramid build of this slot is issued by a later call)
        if (!ql.empty()) VO_TRY(batch_upload_list(B, slot, (int)ql.size(), ql.data(), B->pre_stream));
        const uint8_t* raw = B->q_src[slot];
        if (!B->q_dev[slot]) {
            VO_CUDA(ctx, cudaMemcpyAsync(B->raw_pre.p, B->q_src[slot], ql.empty() ? total : fb * ql.size(), cudaMemcpyHostToDevice,
                                         B->pre_stream));
            raw = (const uint8_t*)B->raw_pre.p;
        }
        if (ql.empty())
            VO_TRY(vo_build_pyramids(ctx, raw, fb, B->cfg.rows, B->cfg.cols, B->geom,
                                     (uint8_t*)B->slabs[B->q_set[slot]].p, B->geom.slab_bytes, B->batch, B->pre_stream, batch_ext_dev(B, 0),
                                     batch_ext_host(B, 0)));
        else
            VO_TRY(vo_build_pyramids(ctx, raw, fb, B->cfg.rows, B->cfg.cols, B->geom, (uint8_t*)B->slabs[B->q_set[slot]].p,
                                     B->geom.slab_bytes, (int)ql.size(), B->pre_stream, batch_ext_dev(B, 0), batch_ext_host(B, 0), 0,
                                     batch_list_row(B, slot), ql.data(), B->batch));
        VO_CUDA(ctx, cudaEventRecord(B->q_ev[slot], B->pre_stream));
        B->q_src[slot] = nullptr;
    }
    return 0;
}

extern "C" int b200vo_batch_prime(b200vo_batch* B, const uint8_t* frames)
{
    if (!B || !frames) return B200VO_E_BADARG;
    b200vo_ctx* ctx = B->ctx;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaStreamSynchronize(B->pre_stream));
    B->q_count = 0;
    VO_TRY(batch_upload_frames(B, frames, B->cur));
    VO_CUDA(ctx, cudaEventRecord(B->step_end_ev, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    B->primed = true;
    return 0;
}

// device-resident core: everything after the new frames are in `frames_dev`
// pyramids of the new frames + KLT for sequences [b0, b0 + nb), enqueued on `stream`
// (frames_dev == nullptr: the pyramids of set B->nxt were built ahead by b200vo_batch_submit_frames)
// which: 0 = pyramids + both point sets in one launch, 1 = landmark set only, 2 = candidate set only, 3 = pyramids only,
// 4 = pyramids + landmark set
static int batch_track(b200vo_batch* B, cudaStream_t stream, int b0, int nb, const uint8_t* frames_dev, const float* lm_pts, const int* n_lm,
                       const float* cand_pts, const int* n_cand, float* lm_next, uint8_t* lm_status, float* cand_next,
                       uint8_t* cand_status, int which = 0)
{
    b200vo_ctx* ctx = B->ctx;
    const b200vo_batch_cfg& c = B->cfg;
    const int nxt = B->nxt;
    const size_t fb = (size_t)c.rows * c.cols, sb = B->geom.slab_bytes;
    const int L = c.max_landmarks, Cn = c.max_candidates;
    if (which == 0 || which == 3 || which == 4) {
        const bool whole = b0 == 0 && nb == B->batch;   // chunked uploads build the pyramids piecewise: no single interval to time
        if (whole) prof_mark(B, 0, stream);
        if (frames_dev && B->step_list)   // the listed images into their sequences' slabs (b0 == 0, nb == batch)
            VO_TRY(vo_build_pyramids(ctx, frames_dev, fb, c.rows, c.cols, B->geom, (uint8_t*)B->slabs[nxt].p, sb, B->step_n, stream,
                                     batch_ext_dev(B, 0), batch_ext_host(B, 0), 0, B->step_list, B->step_list_host, B->batch));
        else if (frames_dev)
            VO_TRY(vo_build_pyramids(ctx, frames_dev + (size_t)b0 * fb, fb, c.rows, c.cols, B->geom,
                                     (uint8_t*)B->slabs[nxt].p + (size_t)b0 * sb, sb, nb, stream, batch_ext_dev(B, b0), batch_ext_host(B, b0)));
        if (whole) { prof_mark(B, 1, stream); B->prof_row_open = B->profile && B->prof_n < B200VO_PROF_RING; }
    }
    KltPointSet sets[2] = {{L, n_lm + b0, lm_pts + (size_t)b0 * L * 2, lm_next + (size_t)b0 * L * 2, lm_status + (size_t)b0 * L, nullptr},
                           {Cn, n_cand + b0, cand_pts + (size_t)b0 * Cn * 2, cand_next + (size_t)b0 * Cn * 2,
                            cand_status + (size_t)b0 * Cn, nullptr}};
    if (which == 3 || (which == 2 && Cn <= 0)) return 0;
    const KltPointSet* first = which == 2 ? sets + 1 : sets;
    const int n_sets = which == 0 ? (Cn > 0 ? 2 : 1) : 1;   // which 1, 4: landmark set; 2: candidate set
    VO_TRY(vo_klt_launch2(ctx, B->geom, (const uint8_t*)B->slabs[B->cur].p + (size_t)b0 * sb, sb,
                          (const uint8_t*)B->slabs[nxt].p + (size_t)b0 * sb, sb, nb, first, n_sets, 0, B->kp, stream, batch_ext_dev(B, b0)));
    return 0;
}

// status==1 compaction, P3P-RANSAC + EPnP, inlier mask -- whole batch, enqueued on `stream`
static int batch_pose(b200vo_batch* B, cudaStream_t stream, const float* lm_obj, const int* n_lm, const float* lm_next, const uint8_t* lm_status,
                      double* pose, uint8_t* pnp_ok, uint8_t* inlier_mask, int* n_inliers)
{
    b200vo_ctx* ctx = B->ctx;
    const b200vo_batch_cfg& c = B->cfg;
    if (B->prof_row_open) prof_mark(B, 2, stream);
    PnpArgs a{};
    a.batch = B->batch; a.cap = c.max_landmarks; a.iters = c.pnp_iters;
    a.obj = B->c_obj; a.img = B->c_img; a.n = B->c_n;
    a.intr = B->intr;
    a.thr_sq = (float)((double)c.pnp_reproj_err * (double)c.pnp_reproj_err);
    a.conf = c.pnp_conf;
    // the ctx's table of cv2 random numbers moves when a longer draw grows it (the bootstrap's E-RANSAC does): look it up
    // at every step rather than keeping the address of creation time (no synchronisation unless it has to grow)
    VO_TRY(vo_rng_table(ctx, B->n_raw, &B->rng));
    a.rng_raw = B->rng; a.n_raw = B->n_raw;
    a.inliers = B->inliers; a.mask = B->c_mask; a.pose = pose;
    vo_pnp_carve_workspace(a, B->pnp_ws);
    a.ok = a.ok_ws;
    static const char* trace_file = getenv("B200VO_TRACE_FILE");   // measurement aid, see batch_write_trace
    if (trace_file) {
        VO_TRY(vo_reserve(ctx, B->trace, (size_t)B->batch * 16 * sizeof(long long)));
        a.phase_clk = (long long*)B->trace.p;
    }
    if (vo_pnp_fused_ok(a, true)) {
        // compaction, RANSAC, EPnP and the mask over the original slots: one CTA per sequence, one launch
        PoseBatchIO io;
        io.n_lm = n_lm; io.lm_next = lm_next; io.lm_status = lm_status; io.lm_obj = lm_obj;
        io.c_orig = B->c_orig; io.mask_out = inlier_mask; io.n_inl_out = n_inliers; io.ok_out = pnp_ok;
        VO_TRY(vo_pnp_fused_launch(ctx, a, io, stream));
    } else {
        compact_tracked_kernel<<<B->batch, 256, 0, stream>>>(c.max_landmarks, n_lm, lm_next, lm_status, lm_obj,
                                                             B->c_obj, B->c_img, B->c_n, B->c_orig);
        ctx->launches++;
        VO_TRY(vo_pnp_launch(ctx, a, true, stream));
        scatter_mask_kernel<<<B->batch, 256, 0, stream>>>(c.max_landmarks, a.ok, a.n_inliers, B->inliers, B->c_orig,
                                                          inlier_mask, n_inliers, pnp_ok);
        ctx->launches++;
    }
    if (B->prof_row_open) { prof_mark(B, 3, stream); B->prof_n++; B->prof_row_open = false; }
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}

// the step's kernels are all enqueued (and joined on the ctx stream): the new frames become the previous ones
int batch_finish(b200vo_batch* B)
{
    VO_CUDA(B->ctx, cudaEventRecord(B->step_end_ev, B->ctx->stream));
    B->cur = B->nxt;
    B->step_list = nullptr; B->step_list_host = nullptr; B->step_n = 0;
    return 0;
}

// Whole-batch step.  The pose chain needs the LANDMARK tracks only, and it is a string of small
// latency-bound kernels, while the tracker fills every SM: landmark tracker + pose chain go to a
// high-priority stream, the candidate tracker to the ctx stream, so that the landmark CTAs are
// dispatched first, the candidate CTAs fill the machine behind them (no idle tail between the two
// launches) and the pose kernels slip in as soon as they are ready.
//   ctx stream:   [pyramids] (pyr_ev) [KLT candidates] (cand_ev) .................... wait(pose_ev)
//   pose stream:       wait(pyr_ev) [KLT landmarks] (lm_ev) [compact][P3P-RANSAC][EPnP][mask] (pose_ev)
int batch_track_pose_overlapped(b200vo_batch* B, const uint8_t* frames_dev, const float* lm_pts, const float* lm_obj,
                                const int* n_lm, const float* cand_pts, const int* n_cand, float* lm_next,
                                uint8_t* lm_status, float* cand_next, uint8_t* cand_status, double* pose,
                                uint8_t* pnp_ok, uint8_t* inlier_mask, int* n_inliers, cudaEvent_t obj_ready,
                                cudaEvent_t cand_ready)
{
    b200vo_ctx* ctx = B->ctx;
    cudaStream_t main_stream = ctx->stream;
    VO_TRY(batch_track(B, main_stream, 0, B->batch, frames_dev, lm_pts, n_lm, cand_pts, n_cand, lm_next, lm_status, cand_next,
                       cand_status, 3));
    VO_CUDA(ctx, cudaEventRecord(B->klt_ev, main_stream));          // pyramids and every input of the step are in place
    VO_CUDA(ctx, cudaStreamWaitEvent(B->pose_stream, B->klt_ev, 0));
    VO_TRY(batch_track(B, B->pose_stream, 0, B->batch, frames_dev, lm_pts, n_lm, cand_pts, n_cand, lm_next, lm_status, cand_next,
                       cand_status, 1));
    VO_CUDA(ctx, cudaEventRecord(B->lm_ev, B->pose_stream));
    if (obj_ready) VO_CUDA(ctx, cudaStreamWaitEvent(B->pose_stream, obj_ready, 0));
    VO_TRY(batch_pose(B, B->pose_stream, lm_obj, n_lm, lm_next, lm_status, pose, pnp_ok, inlier_mask, n_inliers));
    VO_CUDA(ctx, cudaEventRecord(B->pose_ev, B->pose_stream));
    // The tracker is a persistent kernel (one grid fills every SM until its queue is empty): launched beside the
    // landmark set, the candidate set would hold half the machine and the landmark tracks -- which the pose chain
    // waits for -- would take twice as long.  So: landmark set alone, then candidate set and pose chain side by side.
    VO_CUDA(ctx, cudaStreamWaitEvent(main_stream, B->lm_ev, 0));
    if (cand_ready) VO_CUDA(ctx, cudaStreamWaitEvent(main_stream, cand_ready, 0));   // candidate keypoints uploaded beside the landmark tracker
    VO_TRY(batch_track(B, main_stream, 0, B->batch, frames_dev, lm_pts, n_lm, cand_pts, n_cand, lm_next, lm_status, cand_next,
                       cand_status, 2));
    VO_CUDA(ctx, cudaEventRecord(B->cand_ev, main_stream));
    VO_CUDA(ctx, cudaStreamWaitEvent(main_stream, B->pose_ev, 0));
    return 0;
}

int batch_select_frames(b200vo_batch* B, const uint8_t* frames_dev, int n_list, const int32_t* list)
{
    b200vo_ctx* ctx = B->ctx;
    B->step_list = nullptr; B->step_list_host = nullptr; B->step_n = 0;
    if (!frames_dev) {
        // the frames were handed over by b200vo_batch_submit_frames(_dev): their pyramids were (or are being) built on
        // the side stream, beside the previous step
        if (B->q_count == 0)
            return vo_set_err(ctx, B200VO_E_BADARG, "frames == NULL but no frame set was submitted (b200vo_batch_submit_frames[_dev])");
        const int q_slot = B->q_head;
        VO_TRY(batch_issue_prefetch(B));                     // whatever is still waiting, this step's set first
        if (n_list > 0) { B->step_list = batch_list_row(B, q_slot); B->step_list_host = B->q_list[q_slot].data(); B->step_n = n_list; }
        B->nxt = B->q_set[q_slot];
        B->q_head ^= 1;
        B->q_count--;
        VO_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, B->q_ev[q_slot], 0));
    } else {
        if (B->q_count > 0)
            return vo_set_err(ctx, B200VO_E_BADARG, "submitted frame sets are waiting: pass frames == NULL to consume them in order");
        const int free_set = batch_free_set(B);
        if (free_set < 0) return vo_set_err(ctx, B200VO_E_BADARG, "no free pyramid set");
        B->nxt = free_set;
        if (n_list > 0) {   // row 2: the previous step that read it is ordered before this upload on the ctx stream
            VO_TRY(batch_upload_list(B, 2, n_list, list, ctx->stream));
            B->step_list = batch_list_row(B, 2); B->step_list_host = list; B->step_n = n_list;
        }
    }
    return 0;
}

// device-resident core: everything after the new frames are in `frames_dev`
static int batch_core(b200vo_batch* B, const uint8_t* frames_dev, const float* lm_pts, const float* lm_obj,
                      const int* n_lm, const float* cand_pts, const int* n_cand, float* lm_next,
                      uint8_t* lm_status, float* cand_next, uint8_t* cand_status, double* pose, uint8_t* pnp_ok,
                      uint8_t* inlier_mask, int* n_inliers)
{
    b200vo_ctx* ctx = B->ctx;
    if (!B->primed) return vo_set_err(ctx, B200VO_E_BADARG, "b200vo_batch_prime was not called");
    VO_TRY(batch_select_frames(B, frames_dev));
    VO_TRY(batch_track_pose_overlapped(B, frames_dev, lm_pts, lm_obj, n_lm, cand_pts, n_cand, lm_next, lm_status, cand_next,
                                       cand_status, pose, pnp_ok, inlier_mask, n_inliers, nullptr));
    return batch_finish(B);
}

extern "C" int b200vo_batch_step_dev(b200vo_batch* B, const uint8_t* frames_dev, const float* lm_pts_dev,
                                     const float* lm_obj_dev, const int32_t* n_lm_dev, const float* cand_pts_dev,
                                     const int32_t* n_cand_dev, float* lm_next_dev, uint8_t* lm_status_dev,
                                     float* cand_next_dev, uint8_t* cand_status_dev, double* pose_dev,
                                     uint8_t* pnp_ok_dev, uint8_t* inlier_mask_dev, int32_t* n_inliers_dev)
{
    if (!B) return B200VO_E_BADARG;
    VO_CUDA(B->ctx, cudaSetDevice(B->ctx->device));
    return batch_core(B, frames_dev, lm_pts_dev, lm_obj_dev, n_lm_dev, cand_pts_dev, n_cand_dev, lm_next_dev,
                      lm_status_dev, cand_next_dev, cand_status_dev, pose_dev, pnp_ok_dev, inlier_mask_dev,
                      n_inliers_dev);
}

extern "C" int b200vo_batch_step(b200vo_batch* B, const uint8_t* frames, const float* lm_pts, const float* lm_obj,
                                 const int32_t* n_lm, const float* cand_pts, const int32_t* n_cand, float* lm_next,
                                 uint8_t* lm_status, float* cand_next, uint8_t* cand_status, double* pose,
                                 uint8_t* pnp_ok, uint8_t* inlier_mask, int32_t* n_inliers)
{
    if (!B || !lm_pts || !lm_obj || !n_lm || !lm_next || !lm_status || !pose || !pnp_ok || !inlier_mask || !n_inliers)
        return B200VO_E_BADARG;
    b200vo_ctx* ctx = B->ctx;
    const b200vo_batch_cfg& c = B->cfg;
    static const bool host_trace = getenv("B200VO_TRACE_FILE") != nullptr;
    auto now_us = [] { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double h_entry = host_trace ? now_us() : 0;
    double h_in = 0, h_kern = 0, h_rb = 0, h_sync = 0;
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const int nb = B->batch, L = c.max_landmarks, Cn = c.max_candidates;
    const size_t fb = (size_t)c.rows * c.cols, f_total = fb * nb;
    // ---- inputs: frames (direct DMA when the caller's buffer is pinned) + one packed small block ----
    const size_t o_lmp = 0, o_lmo = o_lmp + vo_align((size_t)nb * L * 8, 256), o_nlm = o_lmo + vo_align((size_t)nb * L * 12, 256);
    const size_t o_nc = o_nlm + vo_align((size_t)nb * 4, 256), o_cp = o_nc + vo_align((size_t)nb * 4, 256);   // the two count arrays are adjacent: one DMA
    const size_t in_bytes = o_cp + vo_align((size_t)nb * Cn * 8, 256);
    // ---- outputs packed ----
    const size_t q_lmn = 0, q_lms = q_lmn + vo_align((size_t)nb * L * 8, 256), q_cn = q_lms + vo_align((size_t)nb * L, 256);
    const size_t q_cs = q_cn + vo_align((size_t)nb * Cn * 8, 256), q_pose = q_cs + vo_align((size_t)nb * Cn, 256);
    const size_t q_ok = q_pose + vo_align((size_t)nb * 48, 256), q_mask = q_ok + vo_align((size_t)nb, 256);
    const size_t q_ni = q_mask + vo_align((size_t)nb * L, 256), out_bytes = q_ni + vo_align((size_t)nb * 4, 256);
    VO_TRY(vo_reserve(ctx, B->raw, f_total));
    VO_TRY(vo_reserve(ctx, B->pts_in, in_bytes));
    {   // slots beyond the live counts are never written by the kernels: give them a defined value (0) once
        void* before = B->outs.p;
        VO_TRY(vo_reserve(ctx, B->outs, out_bytes));
        if (B->outs.p != before) VO_CUDA(ctx, cudaMemsetAsync(B->outs.p, 0, out_bytes, ctx->stream));
    }
    if (!B->primed) return vo_set_err(ctx, B200VO_E_BADARG, "b200vo_batch_prime was not called");
    for (int b = 0; b < nb; ++b) {   // the counts are host arrays here: a count beyond the slot capacity is a caller bug
        if (n_lm[b] < 0 || n_lm[b] > L)
            return vo_set_err(ctx, B200VO_E_BADARG, "n_lm[%d] = %d is outside [0, max_landmarks = %d]", b, n_lm[b], L);
        if (Cn > 0 && cand_pts && n_cand && (n_cand[b] < 0 || n_cand[b] > Cn))
            return vo_set_err(ctx, B200VO_E_BADARG, "n_cand[%d] = %d is outside [0, max_candidates = %d]", b, n_cand[b], Cn);
    }
    const bool prefetched = frames == nullptr;
    if (prefetched && B->q_count == 0)
        return vo_set_err(ctx, B200VO_E_BADARG, "frames == NULL but no frame set was submitted (b200vo_batch_submit_frames)");
    if (!prefetched && B->q_count > 0)
        return vo_set_err(ctx, B200VO_E_BADARG, "submitted frame sets are waiting: pass frames == NULL to consume them in order");
    cudaPointerAttributes at{};
    const bool pinned = prefetched || (cudaPointerGetAttributes(&at, frames) == cudaSuccess && at.type == cudaMemoryTypeHost);
    cudaGetLastError();
    VO_TRY(vo_reserve_pinned(ctx, (pinned ? 0 : f_total) + in_bytes + out_bytes));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    const uint8_t* fsrc = frames;
    if (!pinned) { memcpy(hp, frames, f_total); fsrc = hp; hp += f_total; }
    const int q_slot = B->q_head;
    if (prefetched) {
        if (B->q_src[q_slot]) VO_TRY(batch_issue_prefetch(B));   // submitted just now: its copy goes first
        B->nxt = B->q_set[q_slot];
        B->q_head ^= 1;
        B->q_count--;
    } else {
        B->nxt = batch_free_set(B);
        if (B->nxt < 0) return vo_set_err(ctx, B200VO_E_BADARG, "no free pyramid set");
    }
    // Sequences are processed in chunks, each on its own stream: H2D of its frames -> pyramids -> KLT.
    // The copies queue on the DMA engine in order, so chunk k+1 is on the wire while chunk k is tracked,
    // and the long-iteration tail of one chunk's KLT overlaps the next chunk's body.
    const int nchunks = (!prefetched && nb >= 2 * B200VO_BATCH_CHUNKS) ? B200VO_BATCH_CHUNKS : 1;
    const int per = (nb + nchunks - 1) / nchunks;
    // small inputs: page-locked caller arrays are DMA'd in place, pageable ones go through the staging block
    auto is_pinned = [](const void* p) {
        cudaPointerAttributes a{};
        const bool r = p && cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost;
        cudaGetLastError();
        return r;
    };
    uint8_t* di = (uint8_t*)B->pts_in.p;
    auto upload = [&](size_t off, const void* src, size_t bytes, cudaStream_t st) -> cudaError_t {
        if (!src || bytes == 0) return cudaSuccess;
        if (is_pinned(src)) return cudaMemcpyAsync(di + off, src, bytes, cudaMemcpyHostToDevice, st);
        memcpy(hp + off, src, bytes);
        return cudaMemcpyAsync(di + off, hp + off, bytes, cudaMemcpyHostToDevice, st);
    };
    cudaStream_t ms = ctx->stream;
    // Small batches (a single sequence, small shards): the step is latency-bound and a dozen separate DMA operations
    // cost more than the kernels between them.  Pack: one host memcpy per array into the staging block, ONE upload;
    // ONE read-back of the packed result block, host memcpy out.  Large batches keep the in-place DMA of every array.
    const bool packed = in_bytes + out_bytes <= (size_t)B200VO_PACKED_IO_BYTES;
    bool cand_late = false;
    if (packed) {
        memcpy(hp + o_lmp, lm_pts, (size_t)nb * L * 8);
        memcpy(hp + o_lmo, lm_obj, (size_t)nb * L * 12);
        memcpy(hp + o_nlm, n_lm, (size_t)nb * 4);
        if (Cn > 0 && cand_pts && n_cand) {
            memcpy(hp + o_cp, cand_pts, (size_t)nb * Cn * 8);
            memcpy(hp + o_nc, n_cand, (size_t)nb * 4);
        } else {
            memset(hp + o_nc, 0, (size_t)nb * 4);
        }
        VO_CUDA(ctx, cudaMemcpyAsync(di, hp, in_bytes, cudaMemcpyHostToDevice, ms));
        VO_CUDA(ctx, cudaEventRecord(B->done_ev, ctx->stream));
    } else {
    // Only the landmark keypoints and the counts stand between the call and the first kernel (every DMA operation costs
    // 5-8 us of latency on top of its bytes): keypoints in place, both count arrays through the staging block as ONE copy;
    // with prefetched frames the candidate keypoints follow on the io stream (the candidate tracker waits for them),
    // and so do the landmarks, which only PnP needs.
    const bool have_cand = Cn > 0 && cand_pts && n_cand;
    cand_late = have_cand && prefetched;
    VO_CUDA(ctx, upload(o_lmp, lm_pts, (size_t)nb * L * 8, ms));
    memcpy(hp + o_nlm, n_lm, (size_t)nb * 4);
    if (have_cand) memcpy(hp + o_nc, n_cand, (size_t)nb * 4);
    else memset(hp + o_nc, 0, (size_t)nb * 4);
    VO_CUDA(ctx, cudaMemcpyAsync(di + o_nlm, hp + o_nlm, (o_nc - o_nlm) + (size_t)nb * 4, cudaMemcpyHostToDevice, ms));
    if (have_cand && !cand_late) VO_CUDA(ctx, upload(o_cp, cand_pts, (size_t)nb * Cn * 8, ms));
    VO_CUDA(ctx, cudaEventRecord(B->done_ev, ctx->stream));   // points uploaded; previous step fully retired
    if (host_trace) {
        VO_TRY(vo_reserve(ctx, B->stamps, 64 * 4 * 8));
        trace_stamp_kernel<<<1, 1, 0, ctx->stream>>>((unsigned long long*)B->stamps.p + (B->stamp_step & 63) * 4);
    }
    VO_CUDA(ctx, cudaStreamWaitEvent(B->io_stream, B->done_ev, 0));
    if (cand_late) {
        VO_CUDA(ctx, upload(o_cp, cand_pts, (size_t)nb * Cn * 8, B->io_stream));
        VO_CUDA(ctx, cudaEventRecord(B->cand_in_ev, B->io_stream));
    }
    VO_CUDA(ctx, upload(o_lmo, lm_obj, (size_t)nb * L * 12, B->io_stream));
    VO_CUDA(ctx, cudaEventRecord(B->obj_ev, B->io_stream));
    }
    // The copy + pyramid launches of the NEXT frame set (a dozen driver calls, 30-40 us of host time during which the GPU
    // would wait for this step's first kernel) are enqueued after this step's own work instead of in front of it; the copy
    // still queues behind this step's small uploads (done_ev).  The side stream must wait for the PREVIOUS step's end only
    // (the set it overwrites was that step's `cur`), so that wait is enqueued here, before batch_finish re-records the event.
    bool deferred_prefetch = false;
    if (prefetched) {
        for (int k = 0; k < B->q_count; ++k) deferred_prefetch = deferred_prefetch || B->q_src[(B->q_head + k) & 1] != nullptr;
        if (deferred_prefetch) VO_CUDA(ctx, cudaStreamWaitEvent(B->pre_stream, B->step_end_ev, 0));
        VO_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, B->q_ev[q_slot], 0));
    }
    uint8_t* dq = (uint8_t*)B->outs.p;
    cudaStream_t main_stream = ctx->stream;
    if (host_trace) h_in = now_us();
    if (prefetched) {
        // pyramids are already there: landmark tracker, then candidate tracker with the pose chain beside it
        VO_TRY(batch_track_pose_overlapped(B, nullptr, (const float*)(di + o_lmp), (const float*)(di + o_lmo), (const int*)(di + o_nlm),
                                           (const float*)(di + o_cp), (const int*)(di + o_nc), (float*)(dq + q_lmn), dq + q_lms,
                                           (float*)(dq + q_cn), dq + q_cs, (double*)(dq + q_pose), dq + q_ok, dq + q_mask,
                                           (int*)(dq + q_ni), packed ? nullptr : B->obj_ev, cand_late ? B->cand_in_ev : nullptr));
    } else {
        // The frames go up chunk by chunk, back to back on the copy stream; chunk k's pyramids + landmark tracker
        // run on a compute stream as soon as its frames have landed (the later chunks are on the wire meanwhile);
        // its candidate tracker follows on the ctx stream, and the pose chain starts when the last landmark tracks are in.
        if (nchunks > 1) {
            VO_CUDA(ctx, cudaStreamWaitEvent(B->pre_stream, B->step_end_ev, 0));   // B->raw is free again
            VO_CUDA(ctx, cudaStreamWaitEvent(B->pre_stream, B->done_ev, 0));       // behind the step's small uploads
            for (int k = 0; k < nchunks; ++k) {
                const int b0 = k * per, n_here = (b0 + per <= nb ? per : nb - b0);
                if (n_here <= 0) break;
                VO_CUDA(ctx, cudaMemcpyAsync((uint8_t*)B->raw.p + (size_t)b0 * fb, fsrc + (size_t)b0 * fb, (size_t)n_here * fb,
                                             cudaMemcpyHostToDevice, B->pre_stream));
                VO_CUDA(ctx, cudaEventRecord(B->copy_ev[k], B->pre_stream));
            }
        }
        for (int k = 0; k < nchunks; ++k) {
            const int b0 = k * per, n_here = (b0 + per <= nb ? per : nb - b0);
            if (n_here <= 0) break;
            cudaStream_t cs = nchunks > 1 ? B->chunk_stream[k % B200VO_BATCH_STREAMS] : main_stream;
            if (nchunks > 1) VO_CUDA(ctx, cudaStreamWaitEvent(cs, B->copy_ev[k], 0));
            else VO_CUDA(ctx, cudaMemcpyAsync(B->raw.p, fsrc, (size_t)n_here * fb, cudaMemcpyHostToDevice, cs));
            VO_TRY(batch_track(B, cs, b0, n_here, (const uint8_t*)B->raw.p, (const float*)(di + o_lmp), (const int*)(di + o_nlm),
                               (const float*)(di + o_cp), (const int*)(di + o_nc), (float*)(dq + q_lmn), dq + q_lms,
                               (float*)(dq + q_cn), dq + q_cs, 4));
            if (nchunks > 1) {
                VO_CUDA(ctx, cudaEventRecord(B->chunk_ev[k], cs));
                // this chunk's candidates follow on the (normal-priority) ctx stream: they fill the SMs whenever the
                // landmark trackers of later chunks are still waiting for their frames
                VO_CUDA(ctx, cudaStreamWaitEvent(main_stream, B->chunk_ev[k], 0));
                VO_CUDA(ctx, cudaStreamWaitEvent(B->pose_stream, B->chunk_ev[k], 0));
                VO_TRY(batch_track(B, main_stream, b0, n_here, nullptr, (const float*)(di + o_lmp), (const int*)(di + o_nlm),
                                   (const float*)(di + o_cp), (const int*)(di + o_nc), (float*)(dq + q_lmn), dq + q_lms,
                                   (float*)(dq + q_cn), dq + q_cs, 2));
            }
        }
        if (nchunks == 1) {
            VO_CUDA(ctx, cudaEventRecord(B->lm_ev, main_stream));
            VO_CUDA(ctx, cudaStreamWaitEvent(B->pose_stream, B->lm_ev, 0));
            VO_TRY(batch_track(B, main_stream, 0, nb, nullptr, (const float*)(di + o_lmp), (const int*)(di + o_nlm), (const float*)(di + o_cp),
                               (const int*)(di + o_nc), (float*)(dq + q_lmn), dq + q_lms, (float*)(dq + q_cn), dq + q_cs, 2));
        }
        VO_CUDA(ctx, cudaEventRecord(B->cand_ev, main_stream));
        // the pose chain (high priority) starts once every chunk's landmark tracks are done
        if (!packed) VO_CUDA(ctx, cudaStreamWaitEvent(B->pose_stream, B->obj_ev, 0));
        VO_CUDA(ctx, cudaEventRecord(B->lm_ev, B->pose_stream));
        VO_TRY(batch_pose(B, B->pose_stream, (const float*)(di + o_lmo), (const int*)(di + o_nlm), (const float*)(dq + q_lmn),
                          dq + q_lms, (double*)(dq + q_pose), dq + q_ok, dq + q_mask, (int*)(dq + q_ni)));
        VO_CUDA(ctx, cudaEventRecord(B->pose_ev, B->pose_stream));
        VO_CUDA(ctx, cudaStreamWaitEvent(main_stream, B->pose_ev, 0));
    }
    VO_TRY(batch_finish(B));
    if (host_trace) h_kern = now_us();
    uint8_t* ho = hp + in_bytes;
    struct OutCopy { void* dst; size_t off, bytes; bool staged; };
    OutCopy outs[8] = {{lm_next, q_lmn, (size_t)nb * L * 8, false}, {lm_status, q_lms, (size_t)nb * L, false},
                       {Cn > 0 ? cand_next : nullptr, q_cn, (size_t)nb * Cn * 8, false},
                       {Cn > 0 ? cand_status : nullptr, q_cs, (size_t)nb * Cn, false},
                       {pose, q_pose, (size_t)nb * 48, false}, {pnp_ok, q_ok, (size_t)nb, false},
                       {inlier_mask, q_mask, (size_t)nb * L, false}, {n_inliers, q_ni, (size_t)nb * 4, false}};
    if (packed) {
        VO_CUDA(ctx, cudaMemcpyAsync(ho, dq, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        if (deferred_prefetch) VO_TRY(batch_issue_prefetch(B, B->done_ev, false));
        VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
        for (auto& o : outs)
            if (o.dst && o.bytes) memcpy(o.dst, ho + o.off, o.bytes);
        return 0;
    }
    // the tracker's results go home on the io stream while PnP runs; the pose results follow PnP
    VO_CUDA(ctx, cudaStreamWaitEvent(B->io_stream, B->lm_ev, 0));
    for (int i = 0; i < 4; ++i) {
        OutCopy& o = outs[i];
        if (i == 2) {
            VO_CUDA(ctx, cudaStreamWaitEvent(B->io_stream, B->cand_ev, 0));
            if (host_trace && B->stamps.p) trace_stamp_kernel<<<1, 1, 0, B->io_stream>>>((unsigned long long*)B->stamps.p + (B->stamp_step & 63) * 4 + 2);
        }
        if (!o.dst || o.bytes == 0) continue;
        o.staged = !is_pinned(o.dst);
        VO_CUDA(ctx, cudaMemcpyAsync(o.staged ? (void*)(ho + o.off) : o.dst, dq + o.off, o.bytes, cudaMemcpyDeviceToHost, B->io_stream));
    }
    if (host_trace && B->stamps.p) trace_stamp_kernel<<<1, 1, 0, B->io_stream>>>((unsigned long long*)B->stamps.p + (B->stamp_step & 63) * 4 + 3);
    // pose | ok | inlier mask | inlier counts are adjacent in the result block: ONE read-back into the staging block
    // (four DMA operations of a few KB each cost 20-30 us of latency behind the last kernel), host memcpy out
    for (int i = 4; i < 8; ++i) outs[i].staged = true;
    VO_CUDA(ctx, cudaMemcpyAsync(ho + q_pose, dq + q_pose, out_bytes - q_pose, cudaMemcpyDeviceToHost, ctx->stream));
    VO_CUDA(ctx, cudaEventRecord(B->io_ev, B->io_stream));
    VO_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, B->io_ev, 0));
    if (host_trace && B->stamps.p) {
        trace_stamp_kernel<<<1, 1, 0, ctx->stream>>>((unsigned long long*)B->stamps.p + (B->stamp_step & 63) * 4 + 1);
        B->stamp_step++;
    }
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    if (deferred_prefetch) VO_TRY(batch_issue_prefetch(B, B->done_ev, false));
    if (host_trace) h_rb = now_us();
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (host_trace) h_sync = now_us();
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    for (auto& o : outs)
        if (o.dst && o.bytes && o.staged) memcpy(o.dst, ho + o.off, o.bytes);
    if (host_trace) {
        const double h_exit = now_us();
        if (++B->host_calls > 8) {   // the first calls allocate
            B->host_us[0] += h_in - h_entry; B->host_us[1] += h_kern - h_entry; B->host_us[2] += h_rb - h_entry;
            B->host_us[3] += h_sync - h_entry; B->host_us[4] += h_exit - h_entry;
            B->host_us[5] += h_entry - B->host_last_exit;
            B->host_n++;
        }
        B->host_last_exit = h_exit;
    }
    return 0;
}

// cv2.goodFeaturesToTrack (reference :256) on the CURRENT frame of every sequence -- the frames whose pyramids
// the last prime / step left resident -- in one set of launches; no upload, one read-back.
extern "C" int b200vo_batch_good_features(b200vo_batch* B, int max_corners, double quality, double min_dist,
                                          float* corners, int32_t* n_corners)
{
    if (!B || !corners || !n_corners) return B200VO_E_BADARG;
    b200vo_ctx* ctx = B->ctx;
    if (!B->primed) return vo_set_err(ctx, B200VO_E_BADARG, "b200vo_batch_prime was not called");
    VO_CUDA(ctx, cudaSetDevice(ctx->device));
    VO_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    const b200vo_batch_cfg& c = B->cfg;
    const int nb = B->batch;
    if (max_corners <= 0) return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "batched detection needs maxCorners > 0");
    VO_TRY(vo_reserve(ctx, B->gftt_ws, vo_gftt_batch_workspace(c.rows, c.cols, nb, max_corners)));
    float* d_out = nullptr;
    int* d_small = nullptr;
    VO_TRY(vo_gftt_batch_launch(ctx, (const uint8_t*)B->slabs[B->cur].p + B->geom.off[0], B->geom.slab_bytes, B->geom.pitch[0], c.rows, c.cols,
                                nb, max_corners, quality, min_dist, B->gftt_ws.p, &d_out, &d_small, B->ext));
    const size_t b_out = vo_align((size_t)max_corners * 8, 256);
    const size_t out_bytes = b_out * nb, small_bytes = (size_t)nb * VO_GFTT_SMALL * sizeof(int);
    VO_TRY(vo_reserve_pinned(ctx, out_bytes + small_bytes));
    uint8_t* hp = (uint8_t*)ctx->h_pin;
    VO_CUDA(ctx, cudaMemcpyAsync(hp, d_out, out_bytes + small_bytes, cudaMemcpyDeviceToHost, ctx->stream));   // corners | small block are adjacent
    VO_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    VO_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1);
    const int* small = (const int*)(hp + out_bytes);
    for (int s = 0; s < nb; ++s) {
        if (small[s * VO_GFTT_SMALL + 1] > VO_GFTT_BATCH_CAP)
            return vo_set_err(ctx, B200VO_E_UNSUPPORTED, "sequence %d: %d corner candidates exceed the batched path's limit of %d (use the per-image call)",
                              s, small[s * VO_GFTT_SMALL + 1], VO_GFTT_BATCH_CAP);
        const int n = small[s * VO_GFTT_SMALL + 2];
        n_corners[s] = n;
        memcpy(corners + (size_t)s * max_corners * 2, hp + (size_t)s * b_out, (size_t)n * 8);
    }
    return 0;
}

extern "C" int b200vo_batch_profile(b200vo_batch* B, int enable)
{
    if (!B) return B200VO_E_BADARG;
    cudaSetDevice(B->ctx->device);
    if (enable && !B->prof_init) {
        for (auto& row : B->prof_ev) for (auto& e : row) cudaEventCreate(&e);
        B->prof_init = true;
    }
    B->profile = enable != 0;
    B->prof_n = 0;
    B->prof_row_open = false;
    cudaGetLastError();
    return 0;
}

extern "C" int b200vo_batch_profile_read(b200vo_batch* B, float* stage_ms, int* n_steps)
{
    if (!B || !stage_ms || !n_steps) return B200VO_E_BADARG;
    cudaSetDevice(B->ctx->device);
    cudaStreamSynchronize(B->ctx->stream);
    for (int s = 0; s < B200VO_PROF_STAGES; ++s) stage_ms[s] = 0.f;
    for (cudaStream_t st : {B->pose_stream, B->pre_stream}) if (st) cudaStreamSynchronize(st);
    int rows = 0;
    for (int i = 0; i < B->prof_n; ++i) {
        float ms[B200VO_PROF_STAGES];
        bool ok = true;
        for (int s = 0; s < B200VO_PROF_STAGES && ok; ++s)
            ok = cudaEventElapsedTime(&ms[s], B->prof_ev[i][s], B->prof_ev[i][s + 1]) == cudaSuccess;
        if (!ok) { cudaGetLastError(); continue; }   // an incomplete row must not leave a sticky error behind
        for (int s = 0; s < B200VO_PROF_STAGES; ++s) stage_ms[s] += ms[s];
        rows++;
    }
    *n_steps = rows;
    return 0;
}

extern "C" void* b200vo_host_alloc(b200vo_ctx* ctx, size_t bytes)
{
    if (!ctx || bytes == 0) return nullptr;
    cudaSetDevice(ctx->device);
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" void b200vo_host_free(b200vo_ctx* ctx, void* p)
{
    if (!p) return;
    if (ctx) cudaSetDevice(ctx->device);   // ctx == NULL: the context is already gone; page-locked memory is freed all the same
    cudaFreeHost(p);
}
