// Batched SIFT detect + describe (sift.cu), shared with the batched bootstrap (loop.cu).
#pragma once
#include "internal.cuh"

// SIFT of n_frames same-sized frames d_raw + f * raw_stride (tight rows of `cols` bytes), in chunks whose scale spaces fit a
// fixed budget.  Frame f's keypoints, in cv2's order and without duplicates, are rows [d_first_row[f], d_first_row[f] +
// d_n_frame[f]) of ctx->d_sift_out[0] (float32 x, y, size, angle, response, octave as int32 bits: the layout of
// b200vo_sift_detect_and_compute) and, when want_desc, of ctx->d_sift_out[1] (float32 [128]).  Both arrays hold *n_rows rows;
// rows past each frame's count are unused.  Synchronises the ctx stream twice per chunk (extremum and keypoint counts),
// and twice more for a chunk whose rows outgrow the output arrays.
int vo_sift_frames(b200vo_ctx* ctx, const uint8_t* d_raw, size_t raw_stride, int n_frames, int rows, int cols, bool want_desc,
                   int* d_n_frame, int* d_first_row, int* n_rows);
