// The batch object of batch.cu and the helpers the per-frame loop (loop.cu) drives it with.
#pragma once
#include "internal.cuh"

#define B200VO_BATCH_CHUNKS 4
// Streams are a scarce resource: the driver multiplexes them onto 8 hardware queues by default
// (CUDA_DEVICE_MAX_CONNECTIONS) and two streams on one queue serialise.  Chunks share 4 streams.
#define B200VO_BATCH_STREAMS 4
// host-buffer steps whose point arrays and results together stay below this go up / come back as ONE copy each
#define B200VO_PACKED_IO_BYTES (512 * 1024)

// One sequence's settings as the host keeps them (b200vo_batch_set_intrinsics / _frame_size / _detection_mask / _lens);
// the device holds their forms the kernels read (b200vo_batch::intr_buf, ext_buf, mask_buf, dist_buf)
struct VoSeqSettings {
    VoIntrinsics intr;   // K: the camera of the undistorted image
    VoSeqExt ext;
    int model;           // B200VO_LENS_PINHOLE / B200VO_LENS_FISHEYE
    double dist[8];      // pinhole: k1, k2, p1, p2, k3, k4, k5, k6; fisheye: k1 .. k4, 0, 0, 0, 0
    bool raw_set;        // raw: the camera of the raw frames; unset: it is K
    VoIntrinsics raw;
    bool mask;           // has a detection mask
    // the raw frames are undistorted through a map: a fisheye lens, a pinhole coefficient or a raw camera other than K
    bool needs_map() const
    {
        if (model == B200VO_LENS_FISHEYE) return true;
        for (double d : dist)
            if (d != 0.0) return true;
        return raw_set && (raw.fx != intr.fx || raw.fy != intr.fy || raw.cx != intr.cx || raw.cy != intr.cy);
    }
};

struct b200vo_batch {
    b200vo_ctx* ctx;
    int batch;
    b200vo_batch_cfg cfg;
    PyrGeom geom;
    KltParams kp;
    int cur;                 // slab set holding the previous frames
    int nxt;                 // slab set the step in flight tracks into
    DevBuf slabs[3];         // [batch] pyramids each: previous frames, frames being tracked, frames prefetched
    // frames submitted ahead of their step (b200vo_batch_submit_frames): FIFO of at most two slab sets
    int q_set[2]; int q_head = 0, q_count = 0;
    const uint8_t* q_src[2] = {};   // frames whose copy / pyramid build has not been enqueued yet (see batch_issue_prefetch)
    bool q_dev[2] = {};             // q_src is device memory (b200vo_batch_submit_frames_dev): no copy, pyramids straight from it
    // Listed steps (b200vo_loop_step_seqs): a submitted set or a step's frames may cover only the sequences of a list.  Each
    // list lives on the device as a row of 2 * batch ints, [list (n entries) | pos (batch entries: row in the list or -1)]:
    // row 0 / 1 belongs to FIFO slot 0 / 1 (uploaded on the side stream when the set's pyramids are enqueued, after the
    // step that last read the row has ended), row 2 to a step that passes its frames (uploaded on the ctx stream).
    std::vector<int32_t> q_list[2]; // the list a submitted set was given; empty: a full set
    DevBuf lists;                   // [3][2 * batch] int32
    const int* step_list = nullptr; // the device row of the step being enqueued; nullptr: every sequence
    const int32_t* step_list_host = nullptr;
    int step_n = 0;                 // its length
    cudaEvent_t q_ev[2] = {};
    cudaStream_t pre_stream = nullptr;
    cudaEvent_t step_end_ev = nullptr;
    DevBuf raw_pre;          // device copy of the frames being prefetched
    DevBuf raw;              // device copy of the uploaded frames (host-input path)
    DevBuf pts_in;           // host-input path: lm_pts | lm_obj | n_lm | cand_pts | n_cand
    DevBuf outs;             // host-input path: outputs
    DevBuf work;             // compacted landmarks + PnP workspace
    DevBuf gftt_ws;          // batched corner detection workspace
    DevBuf stamps;           // B200VO_TRACE_FILE: GPU wall clock at points of the host-buffer step's streams ([64 steps][4])
    long stamp_step = 0;
    DevBuf trace;            // B200VO_TRACE_FILE: wall-clock stamps of the pose CTAs of the last step ([batch][16] int64)
    double host_us[6] = {};  // B200VO_TRACE_FILE: host time inside b200vo_batch_step, summed: entry->inputs enqueued->kernels enqueued->
    long host_n = 0;         //                    read-back enqueued->synchronised->return, and between two calls
    double host_last_exit = 0;
    long host_calls = 0;
    // carved from `work`
    float* c_obj; float* c_img; int* c_n; int* c_orig; int* inliers; uint8_t* c_mask;
    void* pnp_ws;
    const uint32_t* rng; int n_raw;
    bool primed;
    // the settings of every sequence (batch_apply): the host table, how many sequences have a mask / a map, and the
    // device forms.  intr_buf: the VoIntrinsics rows.  ext_buf: the VoSeqExt rows, read by the pyramid, tracker and detector
    // kernels; `ext` is nullptr while every sequence has the slot size cfg.rows x cfg.cols: the kernels then take the slot
    // geometry from their launch arguments, as a batch without per-sequence sizes always did.  mask_buf: [batch] "has a
    // mask" bytes, then [batch] masks in the slot layout, allocated with the first mask.  dist_buf: [batch] "has a map"
    // bytes, then [batch] int16 source-pixel maps and [batch] uint16 fraction maps in the slot layout (VoUndist), allocated
    // with the first map.  n_mask == 0: the detectors get no mask; n_dist == 0: pyramids as without distortion.
    std::vector<VoSeqSettings> seq;
    int n_mask = 0, n_dist = 0;
    DevBuf intr_buf;
    const VoIntrinsics* intr = nullptr;
    DevBuf ext_buf;
    const VoSeqExt* ext = nullptr;
    DevBuf mask_buf;
    DevBuf dist_buf;
    DevBuf dist_par;                // the parameter rows of the last map build
    // host-input path: frames arrive chunk by chunk on a copy stream while earlier chunks are tracked
    cudaStream_t chunk_stream[B200VO_BATCH_STREAMS] = {};  // chunk k: H2D -> pyramid -> KLT on stream k % STREAMS
    cudaEvent_t chunk_ev[B200VO_BATCH_CHUNKS] = {};
    cudaEvent_t copy_ev[B200VO_BATCH_CHUNKS] = {};   // chunk k's frames have landed (copies run back to back on pre_stream)
    cudaEvent_t done_ev = nullptr;
    cudaStream_t io_stream = nullptr;      // landmark upload / KLT result read-back beside the kernels
    // PnP is a chain of small latency-bound kernels that needs the LANDMARK tracks only: it runs on a
    // high-priority stream beside the candidate tracker (which fills the SMs) instead of after it
    cudaStream_t pose_stream = nullptr;
    cudaEvent_t lm_ev = nullptr, cand_ev = nullptr, pose_ev = nullptr;
    cudaEvent_t obj_ev = nullptr, klt_ev = nullptr, io_ev = nullptr, cand_in_ev = nullptr;
    // optional per-kernel timing (CUDA events on the ctx stream): [step][stage] boundaries
    bool profile = false;
    int prof_n = 0;
    bool prof_row_open = false;   // marks 0 and 1 of row prof_n were recorded by this step
    cudaEvent_t prof_ev[B200VO_PROF_RING][B200VO_PROF_STAGES + 1];
    bool prof_init = false;
};

// the frames of the step about to be enqueued: a submitted set (frames_dev == nullptr) or a free set the step builds
// its pyramids in; sets B->nxt and makes the ctx stream wait for a prefetched set
// With n_list > 0 the step covers the sequences list[0 .. n_list) only (validated by the caller): frames_dev holds their
// images in list order, or the oldest submitted set was submitted with that list; sets step_list / step_n.
int batch_select_frames(b200vo_batch* B, const uint8_t* frames_dev, int n_list = 0, const int32_t* list = nullptr);
// a frame set for a later step; n_list > 0: the images of the sequences list[0 .. n_list) in list order (validated by the caller)
int batch_submit(b200vo_batch* B, const uint8_t* frames, bool dev, int n_list = 0, const int32_t* list = nullptr);
int batch_issue_prefetch(b200vo_batch* B, cudaEvent_t after = nullptr, bool wait_step_end = true);
int batch_free_set(const b200vo_batch* B);
int batch_track_pose_overlapped(b200vo_batch* B, const uint8_t* frames_dev, const float* lm_pts, const float* lm_obj,
                                const int* n_lm, const float* cand_pts, const int* n_cand, float* lm_next,
                                uint8_t* lm_status, float* cand_next, uint8_t* cand_status, double* pose,
                                uint8_t* pnp_ok, uint8_t* inlier_mask, int* n_inliers, cudaEvent_t obj_ready,
                                cudaEvent_t cand_ready = nullptr);
int batch_finish(b200vo_batch* B);
// The setters of the listed sequences' settings: each checks its inputs and, only when all are valid and no submitted frame
// set that depends on the setting waits, waits for the work in flight and applies the new rows (synchronous).  *stale:
// the listed sequences' resident pyramids no longer match their frames (new sizes or maps).
int batch_set_intrinsics(b200vo_batch* B, int n_seq, const int32_t* seqs, const double* K, bool* stale);
int batch_set_frame_size(b200vo_batch* B, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols, bool* stale);
// masks: uint8 [n_seq][cfg.rows][cfg.cols], nullptr: the listed sequences' masks are cleared
int batch_set_detection_mask(b200vo_batch* B, int n_seq, const int32_t* seqs, const uint8_t* masks, bool* stale);
// model: [n_seq] B200VO_LENS_*, nullptr: all pinhole; coeffs: [n_seq][8]; raw_K: [n_seq][9] or nullptr (the raw camera is
// K); a pinhole all-zero row without raw_K clears a sequence's lens
int batch_set_lens(b200vo_batch* B, int n_seq, const int32_t* seqs, const int32_t* model, const double* coeffs, const double* raw_K,
                   bool* stale);
// the masks of the detectors: indexed by sequence, none while no sequence has one
VoMask batch_mask(const b200vo_batch* B);
// the maps of sequences b0 .. b0 + n - 1, or of the n sequences list[k] (b0 == 0); none while none of them needs one
VoUndist batch_undist(const b200vo_batch* B, int b0, int n, const int32_t* list = nullptr);
// The pyramids of n raw images (device, slot layout, one slot apart) into slab set `set`, each at its sequence's extents
// and with its map: image k is sequence b0 + k, or with a list (its device row and host copy, b0 == 0) sequence list[k]
int batch_pyramids(b200vo_batch* B, const uint8_t* raw, int set, int b0, int n, cudaStream_t stream, const int* list_dev = nullptr,
                   const int32_t* list_host = nullptr);
