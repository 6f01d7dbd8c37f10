// Internal declarations shared by the sm_100a kernels and the C-ABI glue of libb200vo.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <vector>
#include "../../include/b200vo.h"

#define VO_MAX_LEVELS 12
#define VO_BORDER 32  // materialised REFLECT_101 border around every pyramid level (pixels)

// One pyramid level of one frame: `base` points at pixel (0,0); rows/cols in
// [-VO_BORDER, dim+VO_BORDER) are valid memory holding the REFLECT_101 extension.
struct PyrLevel {
    uint8_t* base;
    int w, h, pitch;
};
struct Pyramid {
    int levels;
    PyrLevel lv[VO_MAX_LEVELS];
};
// Geometry of a pyramid slab (one frame incl. all levels and borders) -- shared by every
// frame of the same (rows, cols, levels).
struct PyrGeom {
    int levels;
    int w[VO_MAX_LEVELS], h[VO_MAX_LEVELS], pitch[VO_MAX_LEVELS];
    size_t off[VO_MAX_LEVELS];  // byte offset of pixel (0,0) of level l inside the slab
    size_t slab_bytes;
};

// The extents of one sequence's frames inside a batch whose slot (PyrGeom) may be larger: its level count and the
// size of every level by the (w + 1) / 2 chain.  Its image is the top-left w[0] x h[0] of the slot, with the slot's
// row pitch; nothing to the right of or below a level's REFLECT_101 ring is ever read.  A device array of [batch] rows
// per batch object whose sequences do not all have the slot size; kernels given none use the slot's own geometry.
struct VoSeqExt {
    int levels;
    int w[VO_MAX_LEVELS], h[VO_MAX_LEVELS];
};

struct KltParams {
    int win_w, win_h;
    int max_count;
    double eps_sq;     // already squared
    float min_eig_thr;
};

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

struct FrameSlot {
    DevBuf slab;
    PyrGeom geom{};
    int rows = 0, cols = 0;
    bool valid = false;
};

// One sequence's camera as every kernel reads it: a device array of [batch] rows per batch object
// (b200vo_batch_set_intrinsics / b200vo_loop_set_intrinsics), a one-row array for the one-call entry points.  Filled on
// the host by vo_intrinsics_row in exactly the expressions the kernels used when K was a scalar argument, so a sequence
// with a given K sees the same bits whatever the rest of its batch uses.
struct VoIntrinsics {
    double fx, fy, cx, cy;     // K[0], K[4], K[2], K[5]
    double K[9], Ki[9];        // the triangulation's K and its inverse
    float emat_thr_sq;         // E-RANSAC: (float)((thr / ((fx + fy) / 2))^2), Sampson error bound in normalised coordinates
};
#define VO_BOOT_EMAT_THR 1.0   // the bootstrap's findEssentialMat threshold (pixels, :308)

// K is a pinhole camera matrix: fx, fy finite and > 0, cx, cy finite, skew and the other off-diagonal entries 0, last row (0, 0, 1)
bool vo_intrinsics_valid(const double K[9]);
void vo_intrinsics_row(VoIntrinsics& r, const double K[9], double emat_thr);
// The single-K entry points: n identical rows of K in the ctx's own buffer, uploaded on the ctx stream (pageable source,
// staged before the call returns, so the upload never waits for the device)
int vo_intrinsics_uniform(b200vo_ctx* ctx, const double K[9], double emat_thr, int n, const VoIntrinsics** d_rows);
// Validates the n_seq (index, K) pairs of a set_intrinsics call against [0, batch) and fills rows[seqs[k]] of the host mirror
// `rows` ([batch]); nothing is written unless every pair is valid
int vo_intrinsics_set(b200vo_ctx* ctx, int batch, int n_seq, const int32_t* seqs, const double* K, double emat_thr,
                      VoIntrinsics* rows);

struct b200vo_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    char err[1024] = {0};
    long long launches = 0;
    float last_ms = 0.f;
    int num_sms = 148;
    // staging
    DevBuf d_stage_img[2];   // raw uploaded image (tight rows)
    void* h_pin = nullptr;   // pinned host staging
    size_t h_pin_cap = 0;
    DevBuf d_scratch[8];     // generic device scratch (per-API use)
    FrameSlot slots[B200VO_MAX_SLOTS + 2];  // +2 internal slots for the stateless cv2-style call
    int* knn_bad_flag = nullptr;   // device flag of the last kNN call (inside d_scratch[3])
    DevBuf d_klt_queue;      // ring of work-queue counters for the persistent tracker kernel
    unsigned klt_queue_next = 0;
    DevBuf d_sift;           // SIFT scale-space workspace (sift.cu)
    DevBuf d_sift_out[2];    // SIFT keypoints (6 floats a row) and descriptors of the last vo_sift_frames call
    DevBuf d_sift_sort;      // SIFT keypoint sort scratch
    DevBuf d_rng;            // raw cv::RNG stream (uint32)
    int n_rng = 0;
    DevBuf d_intr;           // the one-row intrinsics array of the one-call entry points (vo_intrinsics_one)
    // tensor-map encode entry point (driver API, fetched lazily)
    void* encode_tiled = nullptr;
};

int vo_set_err(b200vo_ctx* ctx, int code, const char* fmt, ...);
int vo_cuda_fail(b200vo_ctx* ctx, cudaError_t e, const char* what);
int vo_reserve(b200vo_ctx* ctx, DevBuf& b, size_t bytes);
int vo_reserve_pinned(b200vo_ctx* ctx, size_t bytes);

#define VO_CUDA(ctx, call)                                         \
    do {                                                           \
        cudaError_t _e = (call);                                   \
        if (_e != cudaSuccess) return vo_cuda_fail(ctx, _e, #call); \
    } while (0)

#define VO_TRY(expr)            \
    do {                        \
        int _rc = (expr);       \
        if (_rc != 0) return _rc; \
    } while (0)

static inline size_t vo_align(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Ordered compaction of [0, n) by one CTA of T threads: emit(i, o) for every i with keep(i), o = its rank among the
// kept ones (what numpy's boolean indexing does).  keep(i) is evaluated once for every i < n.  Returns the count to
// every thread; the trailing barrier makes back-to-back calls safe.
template <int T, class Keep, class Emit>
__device__ __forceinline__ int cta_compact(int n, Keep keep, Emit emit)
{
    __shared__ int s_warp[T / 32];
    __shared__ int s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int base = 0; base < n; base += T) {
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
            for (int w = 0; w < T / 32; ++w) tot += s_warp[w];
            s_base += tot;
        }
        __syncthreads();
    }
    const int r = s_base;
    __syncthreads();
    return r;
}

// ---- pyramid.cu ----
int vo_pyr_levels(int w, int h, int win_w, int win_h, int max_level);
void vo_pyr_geom(int rows, int cols, int levels, PyrGeom* g);
Pyramid vo_pyramid_at(const PyrGeom& g, uint8_t* slab);
// the extents of a rows x cols frame with the level count cv2 builds for it
void vo_seq_ext(int rows, int cols, int win_w, int win_h, int max_level, VoSeqExt* e);
// raw (device, rows of `raw_row` bytes, 0: cols) -> bordered level 0, then levels 1..L-1; `batch` slabs/raws strided.
// d_ext / h_ext: [batch] per-sequence extents on the device and their host copy (both or neither), each inside the
// slot geometry g; every level of a sequence is built at its own size, levels beyond its own count are not built.
// d_list / h_list (both or neither): raw image k goes to slab list[k] of the n_slab slabs at d_slab, with the extents
// ext[list[k]] (the tables then cover all n_slab slabs); the other slabs are not touched.
int vo_build_pyramids(b200vo_ctx* ctx, const uint8_t* d_raw, size_t raw_stride, int rows, int cols,
                      const PyrGeom& g, uint8_t* d_slab, size_t slab_stride, int batch, cudaStream_t stream,
                      const VoSeqExt* d_ext = nullptr, const VoSeqExt* h_ext = nullptr, size_t raw_row = 0,
                      const int* d_list = nullptr, const int* h_list = nullptr, int n_slab = 0);

// ---- gftt.cu: detection on device-resident bordered level-0 images, one per batch entry ----
#define VO_GFTT_SMALL 4          // ints per image in the result block: max bits | n candidates | n corners | spare
#define VO_GFTT_BATCH_CAP 32768  // candidates per image the batched path can rank
size_t vo_gftt_batch_workspace(int rows, int cols, int batch, int max_corners);
// d_ext: [batch] per-sequence extents (level 0 is read), nullptr: every image is rows x cols.  d_list: only the n_img
// images list[k] are detected; their outputs keep the image index (the others' are left stale)
int vo_gftt_batch_launch(b200vo_ctx* ctx, const uint8_t* d_img0, size_t img_stride, int pitch, int rows, int cols, int batch,
                         int max_corners, double quality, double min_dist, void* ws, float** d_corners_out, int** d_small_out,
                         const VoSeqExt* d_ext = nullptr, const int* d_list = nullptr, int n_img = 0);

// ---- klt.cu ----
struct KltPointSet {
    int cap;            // slots per sequence
    const int* n;       // [batch] live points per sequence (device) or nullptr -> n_fixed
    const float* pts;   // [batch][cap][2]
    float* out;         // [batch][cap][2]
    uint8_t* status;    // [batch][cap]
    float* err;         // [batch][cap] or nullptr
};
void vo_klt_trace_read(b200vo_ctx* ctx, std::vector<unsigned long long>& out);   // B200VO_TRACE_FILE aid
// Tracks the points of up to two sets in `batch` independent frame pairs, on `stream`.  d_ext: [batch] per-sequence
// extents (nullptr: every sequence has the geometry g)
int vo_klt_launch2(b200vo_ctx* ctx, const PyrGeom& g, const uint8_t* d_prev_slab, size_t prev_stride,
                   const uint8_t* d_next_slab, size_t next_stride, int batch, const KltPointSet* sets, int n_sets,
                   int n_fixed, const KltParams& kp, cudaStream_t stream, const VoSeqExt* d_ext = nullptr);

// ---- knn.cu: device-resident kNN(k=2) + ratio test on the ctx stream (descriptors float32 [n][128])
size_t vo_knn2_workspace(const b200vo_ctx* ctx, int nq, int nt);   // the scratch vo_knn2_ratio_dev reserves
int vo_knn2_ratio_dev(b200vo_ctx* ctx, const float* q_dev, int nq, const float* t_dev, int nt, double ratio,
                      int* idx2_dev, float* dist2_dev, uint8_t* accept_dev, int* bad_flag_host);
