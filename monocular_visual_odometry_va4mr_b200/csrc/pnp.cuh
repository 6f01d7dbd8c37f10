// Argument block shared by the PnP-RANSAC kernels (all pointers are device memory).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>

struct b200vo_ctx;
struct VoIntrinsics;

struct PnpArgs {
    int batch, cap, iters;
    const float* obj;       // [batch][cap][3]
    const float* img;       // [batch][cap][2]
    const int* n;           // [batch] live correspondences per sequence
    const VoIntrinsics* intr;   // [batch] camera of each sequence (fx, fy, cx, cy)
    float thr_sq;           // (float)(reprojectionError^2)
    double conf;
    const uint32_t* rng_raw;  // raw cv::RNG((uint64)-1) outputs
    int n_raw;
    // workspace
    int* samples;           // [batch][iters][4]   (-1 = no sample)
    double* hyp;            // [batch][iters][12]  R (row-major) | t
    double* hyp_rvec;       // [batch][iters][3]
    int* hyp_ok;            // [batch][iters]
    int* counts;            // [batch][iters]
    int* winner;            // [batch]
    int* iters_run;         // [batch]
    int* n_inliers;         // [batch]
    int* flags;             // [batch] bit0: raw RNG table exhausted
    int* ticket;            // [batch] CTAs of the head scoring pass that have finished
    int* need;              // [batch] hypotheses the replay can still reach after the head chunk
    int h_begin, h_end;     // hypothesis range of this solve/score launch
    int full_counts;        // 1: score every hypothesis (the caller reads counts[]); no early exit
    int head;               // 1: this is the head chunk (computes need[]); 0: tail chunk (honours need[])
    uint8_t* ok_ws;         // [batch] spare per-sequence success flags (callers may point `ok` here)
    long long* phase_clk;   // optional [batch][16] clock64 stamps of the fused kernel's phases (benchmarks/pose_phases.py); usually null
    // outputs
    int* inliers;           // [batch][cap] ascending indices
    uint8_t* mask;          // [batch][cap]
    double* pose;           // [batch][6] rvec | tvec
    uint8_t* ok;            // [batch]
};

// What the batched per-frame step adds around the RANSAC when the whole pose chain runs as ONE kernel
// (pnp_fused_kernel): the status==1 compaction in front (PnpArgs::obj/img/n are then OUTPUTS of the kernel) and the
// inlier mask over the original landmark slots behind.  All null: the correspondences are already compact.
struct PoseBatchIO {
    const int* n_lm = nullptr;            // [batch] live landmark slots
    const float* lm_next = nullptr;       // [batch][cap][2] tracked positions
    const uint8_t* lm_status = nullptr;   // [batch][cap]
    const float* lm_obj = nullptr;        // [batch][cap][3]
    int* c_orig = nullptr;                // [batch][cap] original slot of each compacted correspondence
    uint8_t* mask_out = nullptr;          // [batch][cap] inlier mask over the original slots
    int* n_inl_out = nullptr;             // [batch]
    uint8_t* ok_out = nullptr;            // [batch]
};
#define VO_PNP_FUSED_MAX_N 4096   // correspondences per sequence up to which one CTA runs the whole chain

void vo_rng_raw_stream(uint32_t* out, int n);
bool vo_pnp_fused_ok(const PnpArgs& a, bool gen_samples);
int vo_pnp_fused_launch(b200vo_ctx* ctx, const PnpArgs& a, const PoseBatchIO& io, cudaStream_t stream);
size_t vo_pnp_workspace_bytes(int batch, int cap, int iters);
void vo_pnp_carve_workspace(PnpArgs& a, void* ws);
int vo_pnp_launch(b200vo_ctx* ctx, const PnpArgs& a, bool gen_samples, cudaStream_t stream);
// device table of the raw RNG stream, at least n values (grown on demand, owned by ctx)
int vo_rng_table(b200vo_ctx* ctx, int n, const uint32_t** d_table);
