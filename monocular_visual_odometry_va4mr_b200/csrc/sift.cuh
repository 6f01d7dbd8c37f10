// Batched SIFT detect + describe (sift.cu), shared with the batched bootstrap (loop.cu).
#pragma once
#include "internal.cuh"

// SIFT of n_frames same-sized frames d_raw + f * raw_stride (rows of `row_stride` bytes, 0: tight rows of `cols`), in chunks
// whose scale spaces fit a fixed budget.  Frame f's keypoints, in cv2's order and without duplicates, are rows
// [d_first_row[f], d_first_row[f] + d_n_frame[f]) of ctx->d_sift_out[0] (float32 x, y, size, angle, response, octave as int32
// bits: the layout of b200vo_sift_detect_and_compute) and, when want_desc, of ctx->d_sift_out[1] (float32 [128]).  The rows
// start at row0 (rows [0, row0) of an earlier call are kept); both arrays hold *n_rows rows; rows past each frame's count are
// unused.  Synchronises the ctx stream twice per chunk (extremum and keypoint counts), and twice more for a chunk whose rows
// outgrow the output arrays.
int vo_sift_frames(b200vo_ctx* ctx, const uint8_t* d_raw, size_t raw_stride, int n_frames, int rows, int cols, bool want_desc,
                   int* d_n_frame, int* d_first_row, int* n_rows, int row0 = 0, size_t row_stride = 0);
