// The batch object of batch.cu and the helpers the per-frame loop (loop.cu) drives it with.
#pragma once
#include "internal.cuh"

#define B200VO_BATCH_CHUNKS 4
// Streams are a scarce resource: the driver multiplexes them onto 8 hardware queues by default
// (CUDA_DEVICE_MAX_CONNECTIONS) and two streams on one queue serialise.  Chunks share 4 streams.
#define B200VO_BATCH_STREAMS 4
// host-buffer steps whose point arrays and results together stay below this go up / come back as ONE copy each
#define B200VO_PACKED_IO_BYTES (512 * 1024)

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
    // the camera of every sequence (b200vo_batch_set_intrinsics): device rows read by the kernels, host mirror of them
    DevBuf intr_buf;
    const VoIntrinsics* intr = nullptr;
    std::vector<VoIntrinsics> intr_host;
    // the frame size of every sequence (b200vo_batch_set_frame_size): device rows read by the pyramid, tracker and detector
    // kernels, host mirror of them.  `ext` is nullptr while every sequence has the slot size cfg.rows x cfg.cols: the
    // kernels then take the slot geometry from their launch arguments, as a batch without per-sequence sizes always did.
    DevBuf ext_buf;
    const VoSeqExt* ext = nullptr;
    std::vector<VoSeqExt> ext_host;
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
// Validates the (index, K) pairs and, only when all are valid, waits for the work in flight and uploads the new rows (synchronous)
int batch_set_intrinsics(b200vo_batch* B, int n_seq, const int32_t* seqs, const double* K);
// Validates the (index, rows, cols) triples and, only when all are valid and no submitted frame set waits, waits for the
// work in flight and uploads the new extents (synchronous)
int batch_set_frame_size(b200vo_batch* B, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols);
// the device rows of sequences [b0, ...) and their host copy, or nullptr for both while every sequence has the slot size
inline const VoSeqExt* batch_ext_dev(const b200vo_batch* B, int b0) { return B->ext ? B->ext + b0 : nullptr; }
inline const VoSeqExt* batch_ext_host(const b200vo_batch* B, int b0) { return B->ext ? B->ext_host.data() + b0 : nullptr; }
