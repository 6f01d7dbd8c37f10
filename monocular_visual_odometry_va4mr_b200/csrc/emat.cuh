// Batched five-point essential-matrix RANSAC (emat.cu), shared with the batched bootstrap (loop.cu).
#pragma once
#include "internal.cuh"

// cv2.findEssentialMat(RANSAC) of nseq point sets in one set of launches on the ctx stream.  Set s has n_dev[s] <= max_n <= cap
// points at p1 / p2 + 2 * s * cap (device, float32 pixels) seen by the camera intr_dev[s] (device), whose emat_thr_sq is the
// threshold.  Outputs per set: E_dev[9 * s], mask_dev[s * cap + i] (1 = inlier,
// written for i < n_dev[s]), result_dev[4 * s] = found, iterations run, winner, flags_dev[s] bit 0 = the RNG table ran out
// while drawing subsets (the samples are then not cv2's).  E is written only when found.
int vo_emat_batch(b200vo_ctx* ctx, const float* p1, const float* p2, int cap, const int* n_dev, int max_n, int nseq,
                  const VoIntrinsics* intr_dev, double prob, int max_iters, double* E_dev, uint8_t* mask_dev, int* result_dev,
                  int* flags_dev);
