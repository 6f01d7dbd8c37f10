// Argument blocks of the triangulation kernels (landmarks.cu) and the device-side launchers the per-frame loop
// (loop.cu) uses on its resident state.
#pragma once
#include "internal.cuh"

// one sequence's view of the triangulation kernels, built on the device by tri_sequence
struct TriArgs {
    const double* K; const double* Ki;   // the sequence's K and its inverse (its VoIntrinsics row)
    double cur[12];            // R_CW | t_CW of the current frame (as the reference stores them)
    double min_dist, max_dist, min_angle_deg;
    int min_frames, n, n_poses;
    const float* first_keys; const float* keys; const int* first_pose;
    const double* poses;       // [n_poses][12]
    uint8_t* keep;             // [n] too_short_baseline
    float* lm_slot;            // [n][3] per-candidate result
    float* out_lm; float* out_kp; int* n_new;   // compacted
    int* flags;                // bit0: first_pose out of range
};

// batched forms: blockIdx.y (or blockIdx.x for the compaction) = sequence, ragged counts per sequence
struct TriBatchArgs {
    TriArgs common;            // the gates (the per-sequence fields are filled in by the kernels)
    const VoIntrinsics* intr;  // [batch] camera of each sequence
    int cap, pose_cap;
    const int* n;              // [batch] candidates per sequence
    const int* n_poses;        // [batch]
    const double* cur;         // [batch][12]
    const float* first_keys; const float* keys; const int* first_pose;   // [batch][cap]...
    const double* poses;       // [batch][pose_cap][12]
    uint8_t* keep; float* lm_slot; float* out_lm; float* out_kp; int* n_new; int* flags;   // [batch]...
};

// the reference's gates (main.py:21-25) into the shared part of the argument block
void vo_tri_common(TriArgs& c, double min_dist, double max_dist, double min_angle_deg, int min_frames);
// triangulate_batch_kernel + triangulate_compact_batch_kernel on `stream`; every pointer of `b` is device memory
int vo_triangulate_batch_launch(b200vo_ctx* ctx, const TriBatchArgs& b, int batch, cudaStream_t stream);
// min_distance_batch_kernel on `stream` (valid rows >= n[s] are left as they are)
int vo_min_distance_batch_launch(b200vo_ctx* ctx, int batch, const float* pts, const int* n, int n_cap, const float* existing,
                                 const int* m, int m_cap, float min_dist, uint8_t* valid, cudaStream_t stream);

// cv2.recoverPose for a batch of (E, point set) pairs: sequence s has n[s] <= cap points at p1 / p2 + 2 * s * cap
struct RecArgs {
    const double* E;           // [batch][9]
    const int* valid;          // nullptr or valid[valid_stride * s] != 0: decompose E of sequence s (others keep zero poses)
    int valid_stride;
    const VoIntrinsics* intr;  // [batch] camera of each sequence
    double dist;
    int cap;
    const int* n;              // [batch]
    const float* p1; const float* p2;
    double* poses;             // [batch][4][12] R | t of the four decompositions
    uint8_t* masks;            // nullptr or [batch][4][cap] 0 / 255
    int* good;                 // [batch][4] points passing the cheirality test
    double* Rt;                // [batch][12] the winner's R | t
    int* win;                  // [batch][2] the winner's index and count
};
// decompose, cheirality and winner pick on `stream` (max_n >= every n[s]); every pointer of `a` is device memory
int vo_recover_pose_batch_launch(b200vo_ctx* ctx, const RecArgs& a, int nseq, int max_n, cudaStream_t stream);
