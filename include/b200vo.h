/*
 * b200vo.h -- C ABI of libb200vo.so: the B200 (sm_100a) replacement for the cv2 call
 * sites on the reference's correspondence-and-pose hot path.
 *
 * Each entry point names the reference interface it replaces (file:line in
 * ManuelWendl/Monocular_Visual_Odometry_VA4MR).  Plain pointers and sizes only; all
 * pointers are caller-owned HOST memory unless the function name ends in `_dev`.
 * Return value: 0 = OK; <0 = argument/contract violation (the condition under which cv2
 * raises cv2.error, or B200VO_E_UNSUPPORTED for argument patterns the reference never
 * uses -- there is NO CPU fallback); >0 = CUDA failure (text via b200vo_last_error).
 * Algorithmic non-success (PnP found nothing, KLT lost a point) is not an error.
 *
 * One ctx = one CUDA device + one stream + its buffers; calls on a ctx are serialised by
 * the caller and are synchronous at return (host outputs valid).
 */
#ifndef B200VO_H
#define B200VO_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200vo_ctx b200vo_ctx;

#define B200VO_OK 0
#define B200VO_E_BADARG (-1)      /* cv2.error -215 equivalent */
#define B200VO_E_UNSUPPORTED (-2) /* valid cv2 call, but not a pattern this path implements */
#define B200VO_E_NOMEM (-3)

/* ---- context ---- */
int b200vo_create(int device, b200vo_ctx** out);
void b200vo_destroy(b200vo_ctx* ctx);
const char* b200vo_last_error(b200vo_ctx* ctx);
/* ABI/version probe: returns 100*major+minor; also the compiled sm arch in *sm_arch (e.g. 100). */
int b200vo_version(int* sm_arch);
/* Number of kernels this ctx has launched since creation (bench.py's gpu_launches). */
long long b200vo_launch_count(b200vo_ctx* ctx);
/* Elapsed device time (ms, CUDA events on the ctx stream) of the last API call's GPU work. */
float b200vo_last_gpu_ms(b200vo_ctx* ctx);

/*
 * Replaces cv2.calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, None, winSize=, maxLevel=,
 * criteria=) at VisualOdometryPipeLine.py:281 and :287.
 * prev/next: uint8 rows x cols with row strides in bytes; prev_pts: float32 (n,2).
 * Outputs: next_pts float32 (n,2), status uint8 (n), err float32 (n).
 * crit_type: bit0 = COUNT, bit1 = EPS (cv2.TERM_CRITERIA_*).  flags must be 0.
 */
int b200vo_calc_optical_flow_pyr_lk(b200vo_ctx* ctx, const uint8_t* prev, const uint8_t* next,
                                    int rows, int cols, size_t prev_step, size_t next_step,
                                    const float* prev_pts, int n, int win_w, int win_h,
                                    int max_level, int crit_type, int crit_max_count,
                                    double crit_eps, int flags, double min_eig_thr,
                                    float* next_pts, uint8_t* status, float* err);

/*
 * Frame-slot form of the same call (device-resident pyramids; what the identity-caching
 * shim and the per-frame loop use so that `prev` is not re-uploaded / re-built 4x per frame
 * as cv2 does).  Slots 0..B200VO_MAX_SLOTS-1.
 */
#define B200VO_MAX_SLOTS 4
int b200vo_frame_upload(b200vo_ctx* ctx, int slot, const uint8_t* img, int rows, int cols,
                        size_t step, int win_w, int win_h, int max_level);
int b200vo_klt_slots(b200vo_ctx* ctx, int prev_slot, int next_slot, const float* prev_pts, int n,
                     int win_w, int win_h, int max_level, int crit_type, int crit_max_count,
                     double crit_eps, int flags, double min_eig_thr,
                     float* next_pts, uint8_t* status, float* err);
/* Test hook: copy pyramid level `level` of `slot` (without border) to host (tight rows). */
int b200vo_frame_download_level(b200vo_ctx* ctx, int slot, int level, uint8_t* out, int* w, int* h,
                                int* n_levels);

/*
 * Replaces cv2.goodFeaturesToTrack(img, maxCorners, qualityLevel, minDistance, blockSize=3,
 * useHarrisDetector=False, mask=None) at VisualOdometryPipeLine.py:256.
 * corners_xy: float32 (max_corners,2) caller-allocated; *n_out = corners found (0 -> None).
 */
int b200vo_good_features_to_track(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols,
                                  size_t step, int max_corners, double quality, double min_dist,
                                  int block_size, float* corners_xy, int* n_out);
/*
 * The same with cv2's detection mask (goodFeaturesToTrack(..., mask=)): mask uint8 (rows, cols), `mask_step` bytes a row.
 * A corner needs a nonzero mask byte at its pixel (any nonzero value counts), and the quality threshold is qualityLevel
 * times the largest eigenvalue over the pixels of nonzero bytes only (1-pixel border included), as cv2's
 * minMaxLoc(eig, mask): a masked-out region does not set it.  An all-zero mask gives no corners.  mask == NULL behaves
 * as b200vo_good_features_to_track.  The mask must have the image's size (the caller checks it; cv2 raises otherwise).
 */
int b200vo_good_features_to_track_masked(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols,
                                         size_t step, const uint8_t* mask, size_t mask_step,
                                         int max_corners, double quality, double min_dist,
                                         int block_size, float* corners_xy, int* n_out);

/*
 * Replaces cv2.BFMatcher().knnMatch(desc0, desc1, k=2) at :229 plus the Lowe ratio loop at
 * :218-224.  q (nq,dim), t (nt,dim) float32 row-major, integer-valued 0..255 (SIFT).
 * idx2 int32 (nq,2) (-1 when nt<2), dist2 float32 (nq,2), accept uint8 (nq).
 */
int b200vo_knn2_ratio(b200vo_ctx* ctx, const float* q, int nq, const float* t, int nt, int dim,
                      double ratio, int32_t* idx2, float* dist2, uint8_t* accept);

/*
 * Replaces cv2.findEssentialMat(p1, p2, K, method=RANSAC, prob, threshold) at :308.
 * p1,p2 float32 (n,2); K row-major 3x3.  E row-major 3x3, mask uint8 (n), *found = 0/1.
 */
int b200vo_find_essential_mat_ransac(b200vo_ctx* ctx, const float* p1, const float* p2, int n,
                                     const double K[9], double prob, double thr, int max_iters,
                                     double E[9], uint8_t* mask, int* found);
/*
 * The same RANSAC on the caller's hypothesis sample set (parity runs; the counterpart of
 * b200vo_solve_pnp_ransac_p3p_samples): samples int32 (iters,5).  Every sample is solved and scored;
 * nmodels_out int32 (iters) = models per sample (ascending-root order), counts_out int32 (iters,10) =
 * inliers per (sample, model), models_out double (iters,10,3,3) or NULL, *winner_out = sample * 10 + model
 * as cv2's sequential loop picks it (-1: none), *iters_run = iterations that loop executes.
 */
int b200vo_find_essential_mat_ransac_samples(b200vo_ctx* ctx, const float* p1, const float* p2, int n,
                                             const double K[9], const int32_t* samples, int iters,
                                             double prob, double thr, double E[9], uint8_t* mask,
                                             int* found, int32_t* nmodels_out, int32_t* counts_out,
                                             double* models_out, int* winner_out, int* iters_run);

/*
 * ---- device-pointer forms of the five call sites (SURVEY.md 8b "_dev") ----
 * Same arguments with every array already resident in DEVICE memory (e.g. torch data_ptr()) and the
 * results left there; asynchronous on the ctx stream (b200vo_stream / b200vo_sync).  The counts that
 * the host forms return by value come back as one-element device arrays.
 */
int b200vo_calc_optical_flow_pyr_lk_dev(b200vo_ctx* ctx, const uint8_t* prev_dev, const uint8_t* next_dev,
                                        int rows, int cols, size_t prev_step, size_t next_step,
                                        const float* prev_pts_dev, int n, int win_w, int win_h,
                                        int max_level, int crit_type, int crit_max_count,
                                        double crit_eps, int flags, double min_eig_thr,
                                        float* next_pts_dev, uint8_t* status_dev, float* err_dev);
/* corners_dev float32 (max_corners,2); n_out_dev int32[1] (-1: more than 32768 candidates above the
 * quality threshold -- use the host form).  Needs minDistance >= 1 and maxCorners > 0. */
int b200vo_good_features_to_track_dev(b200vo_ctx* ctx, const uint8_t* img_dev, int rows, int cols,
                                      size_t step, int max_corners, double quality, double min_dist,
                                      int block_size, float* corners_dev, int32_t* n_out_dev);
/* bad_dev (may be NULL) int32[1]: 1 when a descriptor is not integer-valued in 0..255. */
int b200vo_knn2_ratio_dev(b200vo_ctx* ctx, const float* q_dev, int nq, const float* t_dev, int nt,
                          int dim, double ratio, int32_t* idx2_dev, float* dist2_dev,
                          uint8_t* accept_dev, int32_t* bad_dev);
/* E_dev double[9], mask_dev uint8 (n), found_dev int32[1]. */
int b200vo_find_essential_mat_ransac_dev(b200vo_ctx* ctx, const float* p1_dev, const float* p2_dev,
                                         int n, const double K[9], double prob, double thr,
                                         int max_iters, double* E_dev, uint8_t* mask_dev,
                                         int32_t* found_dev);
/* pose_dev double[6] = rvec | tvec, inliers_dev int32 (n), n_inliers_dev int32[1], success_dev uint8[1]. */
int b200vo_solve_pnp_ransac_p3p_dev(b200vo_ctx* ctx, const float* obj_dev, const float* img_dev, int n,
                                    const double K[9], int iters, float reproj_err, double conf,
                                    double* pose_dev, int32_t* inliers_dev, int32_t* n_inliers_dev,
                                    uint8_t* success_dev);

/* Measurement aid: b200vo_solve_pnp_ransac_p3p_dev with the fused pose kernel's phase stamps (SM clock of thread 0
 * at its phase boundaries, see pnp.cu) returned in clk_host[16]; kernel_ms = CUDA-event time of the launch. */
int b200vo_debug_pose_phases(b200vo_ctx* ctx, const float* obj_dev, const float* img_dev, int n,
                             const double K[9], int iters, float reproj_err, double conf,
                             long long* clk_host, float* kernel_ms);

/*
 * ---- components next to the hot path (SURVEY.md 8f) ----
 *
 * Replaces the candidate min-distance filter of feature_adding at :258
 *   valid_dist[i] = np.all(np.linalg.norm(pts[i,:] - self.potential_keys, axis=1) > min_dist)
 * pts float32 (n,2) = the goodFeaturesToTrack corners, existing float32 (m,2) = potential_keys;
 * valid uint8 (n).  float32 arithmetic rounded as numpy rounds it (m == 0: all valid).
 */
int b200vo_min_distance_mask(b200vo_ctx* ctx, const float* pts, int n, const float* existing, int m,
                             float min_dist, uint8_t* valid);

/*
 * Replaces the per-candidate loop of triangulate_landmarks at :107-206: age gate (:171-174),
 * bearing-angle gate check_baseline (:117-147), cv2.triangulatePoints (:188-193), float32
 * de-homogenisation (:194) and the depth window disambguate_landmark (:149-168).
 * first_keys / keys float32 (n,2) = potential_first_keys / potential_keys; first_pose int32 (n) =
 * potential_transforms; poses_cw double (n_poses,12) = self.transforms as (R_CW row-major | t_CW),
 * n_poses = len(self.transforms) at call time; cur_pose_cw = (R_current_CW | t_current_CW).
 * too_short_baseline uint8 (n) is the mask the reference hands to filter_potential (:206);
 * new_landmarks float32 (*n_new,3) / new_keypoints float32 (*n_new,2) are the rows it appends to
 * matched_landmarks / matched_keypoints, in candidate order (caller provides room for n rows).
 */
int b200vo_triangulate_landmarks(b200vo_ctx* ctx, const double K[9], double min_dist, double max_dist,
                                 double min_baseline_angle_deg, int min_baseline_frames,
                                 const float* first_keys, const float* keys, const int32_t* first_pose,
                                 int n, const double* poses_cw, int n_poses,
                                 const double cur_pose_cw[12], uint8_t* too_short_baseline,
                                 float* new_landmarks, float* new_keypoints, int* n_new);
/*
 * Batched forms of the two components above ("batched f1/f2 on the resident batch state", SURVEY.md 8f): the same
 * per-sequence work for every sequence of a batch, one or two launches for the whole batch.  Arrays carry a leading
 * batch axis and a fixed capacity per sequence; n / m / n_poses give the live rows of each sequence.
 *   pts (batch,n_cap,2), existing (batch,m_cap,2) float32 -> valid uint8 (batch,n_cap) (rows >= n[s] are 0).
 *   first_keys / keys (batch,cap,2) float32, first_pose (batch,cap) int32, poses_cw (batch,pose_cap,12) double,
 *   cur_pose_cw (batch,12) double -> too_short_baseline uint8 (batch,cap), new_landmarks (batch,cap,3) and
 *   new_keypoints (batch,cap,2) float32 compacted per sequence, n_new int32 (batch).
 */
int b200vo_batch_min_distance_mask(b200vo_ctx* ctx, int batch, const float* pts, const int32_t* n, int n_cap,
                                   const float* existing, const int32_t* m, int m_cap, float min_dist,
                                   uint8_t* valid);
int b200vo_batch_triangulate_landmarks(b200vo_ctx* ctx, const double K[9], double min_dist, double max_dist,
                                       double min_baseline_angle_deg, int min_baseline_frames, int batch,
                                       int cap, const float* first_keys, const float* keys,
                                       const int32_t* first_pose, const int32_t* n, const double* poses_cw,
                                       const int32_t* n_poses, int pose_cap, const double* cur_pose_cw,
                                       uint8_t* too_short_baseline, float* new_landmarks,
                                       float* new_keypoints, int32_t* n_new);

/*
 * Replaces cv2.recoverPose(E, points1, points2, K) at :315 (default distanceThresh = 50):
 * decomposeEssentialMat + cheirality test of the four (R, +-t) on triangulated points.
 * E row-major 3x3; p1, p2 float32 (n,2) pixels; R row-major 3x3, t (3); mask uint8 (n), 0 / 255 as
 * cv2 writes it; *n_good = cv2's return value (points passing the test for the chosen pose).
 */
int b200vo_recover_pose(b200vo_ctx* ctx, const double E[9], const float* p1, const float* p2, int n,
                        const double K[9], double distance_thresh, double R[9], double t[3],
                        uint8_t* mask, int* n_good);

/*
 * Replaces cv2.SIFT_create().detectAndCompute(img, None) at :35, :226-227 (SURVEY.md 8f row f4; default parameters:
 * nfeatures 0, nOctaveLayers 3, contrastThreshold 0.04, edgeThreshold 10, sigma 1.6, image doubled, float32 descriptors).
 * img uint8 (rows, cols), `step` bytes per row.  kps float32 (max_kp, 6): x, y, size, angle, response and the bits of
 * cv2's packed int32 `octave` field, in cv2's output order (KeyPointsFilter::removeDuplicatedSorted); desc float32
 * (max_kp, 128), integer-valued 0..255, or NULL.  *n_out = keypoints found; only the first max_kp are written.
 */
int b200vo_sift_detect_and_compute(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols, size_t step, int max_kp,
                                   float* kps, float* desc, int32_t* n_out);
/*
 * The same with cv2's detection mask (detectAndCompute(img, mask)): mask uint8 (rows, cols), `mask_step` bytes a row.  As
 * cv2's KeyPointsFilter::runByPixelsMask after the duplicate removal, a keypoint is dropped when the mask byte at
 * ((int)(y + 0.5f), (int)(x + 0.5f)) is 0; the others keep their order and descriptors, and *n_out counts them.
 * mask == NULL behaves as b200vo_sift_detect_and_compute.  The mask must have the image's size (cv2 does not check it).
 */
int b200vo_sift_detect_and_compute_masked(b200vo_ctx* ctx, const uint8_t* img, int rows, int cols, size_t step,
                                          const uint8_t* mask, size_t mask_step, int max_kp, float* kps,
                                          float* desc, int32_t* n_out);
/*
 * Replaces cv2.undistort(src, K, dist) (newCameraMatrix = K): src uint8 (rows, cols), `step` bytes a row; dst uint8
 * (rows, cols), tight.  K a pinhole camera matrix (as b200vo_batch_set_intrinsics accepts); dist double [n_dist], n_dist
 * 4 (k1, k2, p1, p2), 5 (+ k3) or 8 (+ k4, k5, k6, the rational model), all finite.  Byte for byte what cv2 computes: the
 * map of initUndistortRectifyMap(..., CV_16SC2) (1/32 px) and a fixed-point bilinear remap with BORDER_CONSTANT 0, so
 * pixels that map outside the image (or to a non-finite point) are 0.  Other n_dist: B200VO_E_UNSUPPORTED.
 */
int b200vo_undistort(b200vo_ctx* ctx, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                     const double* dist, int n_dist, uint8_t* dst);
/*
 * Replaces cv2.undistort(src, K, dist, newCameraMatrix=Knew): as b200vo_undistort, with the undistorted image seen by the
 * pinhole camera Knew (e.g. from cv2.getOptimalNewCameraMatrix) instead of K.  Knew == K is b200vo_undistort.
 */
int b200vo_undistort_new_camera(b200vo_ctx* ctx, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                                const double* dist, int n_dist, const double Knew[9], uint8_t* dst);
/* Lens models of the per-sequence lens (b200vo_batch_set_lens) */
#define B200VO_LENS_PINHOLE 0   /* cv2's polynomial / rational model: k1, k2, p1, p2, k3, k4, k5, k6 */
#define B200VO_LENS_FISHEYE 1   /* cv2.fisheye's equidistant model: k1, k2, k3, k4 */
/*
 * Replaces cv2.fisheye.undistortImage(src, K, D, Knew=Knew): src uint8 (rows, cols), `step` bytes a row; dst uint8 (rows,
 * cols), tight.  K and Knew pinhole camera matrices, Knew == NULL the identity (as in cv2; usually the caller passes K or
 * cv2.fisheye.estimateNewCameraMatrixForUndistortRectify's matrix); D double [4], finite.  Byte for byte what cv2
 * computes: the map of cv2.fisheye.initUndistortRectifyMap(K, D, I, Knew, size, CV_16SC2), whose source pixel wraps
 * modulo 2^16 as cv2 stores it, and a fixed-point bilinear remap with BORDER_CONSTANT 0.
 */
int b200vo_fisheye_undistort(b200vo_ctx* ctx, const uint8_t* src, int rows, int cols, size_t step, const double K[9],
                             const double D[4], const double* Knew, uint8_t* dst);

/*
 * Replaces cv2.solvePnPRansac(obj, img, K, zeros(4), flags=SOLVEPNP_P3P, confidence=,
 * reprojectionError=, iterationsCount=) at :343 (incl. cv2's EPnP refit on the inliers).
 * obj float32 (n,3), img float32 (n,2).  inliers int32 (n) caller-allocated, ascending,
 * *n_inliers valid entries.  *success = 0 -> rvec/tvec unspecified, n_inliers = 0.
 */
int b200vo_solve_pnp_ransac_p3p(b200vo_ctx* ctx, const float* obj, const float* img, int n,
                                const double K[9], int iters, float reproj_err, double conf,
                                double rvec[3], double tvec[3], int32_t* inliers, int* n_inliers,
                                int* success);
/* Same, but with the hypothesis sample set supplied by the caller (parity tests: "same
 * hypothesis sample set"): samples int32 (iters,4). */
int b200vo_solve_pnp_ransac_p3p_samples(b200vo_ctx* ctx, const float* obj, const float* img, int n,
                                        const double K[9], const int32_t* samples, int iters,
                                        float reproj_err, double conf, double rvec[3],
                                        double tvec[3], int32_t* inliers, int* n_inliers,
                                        int* success, int32_t* counts_out /* iters or NULL */,
                                        int* winner_iter, int* iters_run);

/*
 * Batched per-frame hot path for independent sequences (BASELINE config 5): for each of
 * `batch` sequences, KLT on the landmark keypoints and on the candidate keypoints
 * (:281,:287) from the sequence's previous frame (kept resident from the previous step) to
 * its new frame, then P3P-RANSAC + EPnP on the tracked landmarks (:343).
 * Host arrays are [batch]-major; see INTEGRATION.md for the exact layout.
 */
typedef struct b200vo_batch b200vo_batch;
typedef struct {
    int rows, cols;
    int win_w, win_h, max_level, crit_type, crit_max_count;
    double crit_eps, min_eig_thr;
    int pnp_iters;
    float pnp_reproj_err;
    double pnp_conf;
    double K[9];
    int max_landmarks;  /* capacity per sequence */
    int max_candidates; /* capacity per sequence */
} b200vo_batch_cfg;

int b200vo_batch_create(b200vo_ctx* ctx, int batch, const b200vo_batch_cfg* cfg, b200vo_batch** out);
void b200vo_batch_destroy(b200vo_batch* b);
/*
 * Per-sequence camera intrinsics.  b200vo_batch_create gives every sequence cfg->K; this call gives each of the n_seq distinct
 * sequences seqs[k] the camera matrix K[k] (double [n_seq][9], row-major), which the pose chain of every later step uses.
 * K[k] must be a pinhole camera: fx, fy finite and > 0, cx, cy finite, skew and the other off-diagonal entries 0, last row
 * (0, 0, 1).  Bad indices (out of range, repeated), n_seq < 1, null arrays or a bad K: B200VO_E_BADARG and nothing changes.
 * Synchronous (waits for the step in flight); touches nothing but the listed sequences' intrinsics.
 */
int b200vo_batch_set_intrinsics(b200vo_batch* b, int n_seq, const int32_t* seqs, const double* K);
/*
 * Per-sequence frame size.  cfg->rows x cfg->cols is the size of a SLOT, the largest frame the batch accepts, and every
 * frame array keeps the slot layout [batch][cfg->rows][cfg->cols].  b200vo_batch_create gives every sequence the slot size;
 * this call gives each of the n_seq distinct sequences seqs[k] the frame size rows[k] x cols[k] (int32 [n_seq]): its image
 * is the top-left rows[k] x cols[k] of its slot (row stride cfg->cols), the bytes to the right of and below it are never
 * read, and it is tracked and detected exactly as in a batch of its own size (its own pyramid level count included).
 * A size must fit the slot and be larger than the window (cfg->win_h x cfg->win_w).  Bad indices (out of range, repeated),
 * n_seq < 1, null arrays, a bad size or submitted frame sets still waiting: B200VO_E_BADARG and nothing changes.
 * The resident frames no longer match: the next step needs b200vo_batch_prime.  The listed sequences' detection masks
 * are cleared (a mask has its sequence's frame size).  Synchronous.
 */
int b200vo_batch_set_frame_size(b200vo_batch* b, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols);
/*
 * Per-sequence detection mask (cv2's goodFeaturesToTrack(..., mask=)), for static regions whose corners move with the
 * camera: a car's hood, the black wedges of an undistorted image, a burned-in timestamp or logo.  masks: uint8
 * [n_seq][cfg->rows][cfg->cols] in the slot layout; sequence seqs[k]'s mask is the top-left of row k at its own frame size
 * (bytes outside it are never read).  b200vo_batch_good_features then detects in that sequence exactly as
 * b200vo_good_features_to_track_masked on its frame and mask.  masks == NULL clears the listed sequences' masks.  The mask
 * gates detection only: tracking and pose do not read it.  Bad indices (out of range, repeated), n_seq < 1 or a null seqs:
 * B200VO_E_BADARG and nothing changes.  The mask memory (batch x rows x cols bytes) is allocated with the first mask; a
 * batch without masks runs the detector without mask reads.  Synchronous (waits for the step in flight).  Unlike a frame
 * size, a mask may change while submitted frame sets wait: it applies to every step that runs after the call, those sets'
 * steps included, as the frames' pyramids do not depend on it.
 */
int b200vo_batch_set_detection_mask(b200vo_batch* b, int n_seq, const int32_t* seqs, const uint8_t* masks);
/*
 * Per-sequence lens distortion.  dist: double [n_seq][8], k1, k2, p1, p2, k3, k4, k5, k6 (cv2's order; pad shorter models
 * with zeros); an all-zero row clears a sequence's distortion.  Every frame handed to the batch is raw camera output: a
 * sequence with distortion has its level 0 built from cv2.undistort(frame, K, dist) (b200vo_undistort, newCameraMatrix =
 * K), gathered on the device while the pyramid is built, so points, poses and detection masks are all in the undistorted
 * image, whose camera is the sequence's K.  The map is a function of K, the coefficients and the frame size: this call,
 * b200vo_batch_set_intrinsics and b200vo_batch_set_frame_size rebuild it for the sequences with distortion (the
 * coefficients survive a frame-size change).  Bad indices (out of range, repeated), n_seq < 1, null arrays, a non-finite
 * coefficient or submitted frame sets still waiting: B200VO_E_BADARG and nothing changes.  The resident frames no longer
 * match: the next step needs b200vo_batch_prime.  While submitted frame sets wait, b200vo_batch_set_intrinsics refuses a
 * sequence with distortion too.  The map memory (6 bytes a slot pixel per sequence) is allocated with the first
 * distortion; a batch without distortion builds its pyramids as it always did.  Synchronous.
 */
int b200vo_batch_set_distortion(b200vo_batch* b, int n_seq, const int32_t* seqs, const double* dist);
/*
 * Per-sequence lens: b200vo_batch_set_distortion generalised to fisheye lenses and to raw cameras other than K.
 * model: int32 [n_seq], B200VO_LENS_PINHOLE or B200VO_LENS_FISHEYE, or NULL: every row pinhole.  coeffs: double
 * [n_seq][8], pinhole in cv2's order as b200vo_batch_set_distortion, fisheye k1, k2, k3, k4 in slots 0-3 and zeros in
 * slots 4-7.  raw_K: double [n_seq][9], the
 * pinhole camera the raw frames come from (the one the coefficients belong to), or NULL: the raw camera is the sequence's
 * K.  The sequence's K (b200vo_batch_set_intrinsics) stays the camera of the undistorted image, which is what points,
 * poses, masks and the bootstrap see: cv2.undistort(frame, raw_K, coeffs, newCameraMatrix=K) or
 * cv2.fisheye.undistortImage(frame, raw_K, coeffs, Knew=K).  A sequence needs a map when it is fisheye (all-zero
 * coefficients are the equidistant projection, not the identity), has a nonzero pinhole coefficient, or has a raw camera
 * other than K; a pinhole row of zeros with raw_K NULL clears its lens.  b200vo_batch_set_intrinsics changes K and keeps
 * an explicit raw camera; both it and b200vo_batch_set_frame_size rebuild the map.  b200vo_batch_set_distortion(dist) is
 * this call with model NULL and raw_K NULL.  Bad indices (out of range, repeated), n_seq < 1, a null seqs or coeffs, an
 * unknown model, a non-finite coefficient, a fisheye row with nonzero slots 4-7, a raw_K that is not a pinhole camera
 * matrix, or submitted frame sets still waiting: B200VO_E_BADARG and nothing changes.  The resident frames no longer
 * match: the next step needs b200vo_batch_prime.  Synchronous.
 */
int b200vo_batch_set_lens(b200vo_batch* b, int n_seq, const int32_t* seqs, const int32_t* model, const double* coeffs,
                          const double* raw_K);
/* Upload the first frame of every sequence (frames: batch x rows x cols, tight). */
int b200vo_batch_prime(b200vo_batch* b, const uint8_t* frames);
/*
 * One step.  frames: batch x rows x cols uint8 (new frame per sequence).
 * lm_pts float32 (batch,max_landmarks,2), lm_obj float32 (batch,max_landmarks,3), n_lm int32 (batch);
 * cand_pts float32 (batch,max_candidates,2), n_cand int32 (batch).
 * Outputs: lm_next/lm_status/cand_next/cand_status shaped like the inputs;
 * pose double (batch,6) = rvec|tvec; pnp_ok uint8 (batch); inlier_mask uint8 (batch,max_landmarks)
 * over the landmark slots (0 for untracked); n_inliers int32 (batch).
 * The new frame becomes the sequence's previous frame for the next step.
 * frames == NULL consumes the oldest frame set handed over by b200vo_batch_submit_frames.
 * Page-locked arrays (b200vo_host_alloc) are DMA'd in place; pageable ones are staged.
 */
int b200vo_batch_step(b200vo_batch* b, const uint8_t* frames, const float* lm_pts,
                      const float* lm_obj, const int32_t* n_lm, const float* cand_pts,
                      const int32_t* n_cand, float* lm_next, uint8_t* lm_status, float* cand_next,
                      uint8_t* cand_status, double* pose, uint8_t* pnp_ok, uint8_t* inlier_mask,
                      int32_t* n_inliers);
/*
 * Frames of a FUTURE step (a video reader knows them before the tracker needs them): the copy to
 * the device and the pyramid build run on a side stream and overlap the kernels of the step in
 * flight.  frames must be page-locked (b200vo_host_alloc) and stay untouched until the step that
 * consumes them (b200vo_batch_step with frames == NULL) has returned.  At most two sets may wait.
 */
int b200vo_batch_submit_frames(b200vo_batch* b, const uint8_t* frames);
/* The same look-ahead for frames that are already resident and complete in device memory: no copy,
 * the pyramids are built from frames_dev on the side stream beside the step in flight.  Consumed
 * by b200vo_batch_step_dev (or b200vo_batch_step) with frames == NULL, oldest first. */
int b200vo_batch_submit_frames_dev(b200vo_batch* b, const uint8_t* frames_dev);
/* Same step with every input already resident in device memory and outputs left there
 * (bench.py `value`: no host<->device copies in the timed region).  Asynchronous on the
 * ctx stream; pair with b200vo_sync.  frames_dev == NULL consumes the oldest submitted frame set. */
int b200vo_batch_step_dev(b200vo_batch* b, const uint8_t* frames_dev, const float* lm_pts_dev,
                          const float* lm_obj_dev, const int32_t* n_lm_dev,
                          const float* cand_pts_dev, const int32_t* n_cand_dev, float* lm_next_dev,
                          uint8_t* lm_status_dev, float* cand_next_dev, uint8_t* cand_status_dev,
                          double* pose_dev, uint8_t* pnp_ok_dev, uint8_t* inlier_mask_dev,
                          int32_t* n_inliers_dev);
/*
 * cv2.goodFeaturesToTrack (:256) on the CURRENT frame of every sequence of the batch (the frames the last
 * prime / step made resident): no upload, one set of launches, one read-back.  corners float32
 * (batch, max_corners, 2) in cv2's order, n_corners int32 (batch).  blockSize 3, no mask, no Harris;
 * needs min_dist >= 1 and max_corners > 0 (what the reference passes); more than 32768 candidates above
 * the quality threshold in one image -> B200VO_E_UNSUPPORTED (use b200vo_good_features_to_track).
 */
int b200vo_batch_good_features(b200vo_batch* b, int max_corners, double quality, double min_dist,
                               float* corners, int32_t* n_corners);
/* Per-stage device timing of batch steps (CUDA events on the ctx stream).  Stages:
 * 0 = pyramid build, 1 = KLT kernel, 2 = compaction + PnP-RANSAC + EPnP + mask scatter. */
#define B200VO_PROF_STAGES 3
#define B200VO_PROF_RING 512
int b200vo_batch_profile(b200vo_batch* b, int enable);
/* Sums the recorded stage times (ms) over the *n_steps profiled steps since the last enable. */
int b200vo_batch_profile_read(b200vo_batch* b, float* stage_ms /* [B200VO_PROF_STAGES] */, int* n_steps);
/*
 * ---- the whole per-frame loop on the device (INTEGRATION.md 3d) ----
 * `continuous_operation` (:326-373) for `batch` independent sequences with the VO state of every sequence resident in
 * device memory.  One step tracks the landmarks and the candidates into the new frame, runs P3P-RANSAC + EPnP, keeps
 * the inliers, triangulates the candidates, detects new corners, appends the candidates that pass the distance
 * filter and the new pose.  Only a small result block per sequence leaves the device.
 * A sequence that cannot follow the reference's data flow stops with a status code and is skipped (its state is
 * left as it is) until it is loaded again.
 */
typedef struct b200vo_loop b200vo_loop;
typedef struct {
    b200vo_batch_cfg batch;          /* tracker + PnP; max_landmarks / max_candidates = state capacities per sequence */
    double min_dist_landmarks, max_dist_landmarks, min_baseline_angle_deg;   /* main.py:21-25 */
    int min_baseline_frames;
    int max_corners;                 /* goodFeaturesToTrack (main.py:28-33): blockSize 3, no mask, no Harris */
    double quality_level, feature_min_dist;
    int max_frames;                  /* pose-history capacity per sequence */
} b200vo_loop_cfg;

#define B200VO_LOOP_OK 0
#define B200VO_LOOP_IDLE 1          /* never loaded */
#define B200VO_LOOP_FEW_POINTS 2    /* fewer than 8 landmarks tracked (:342) */
#define B200VO_LOOP_PNP_FAILED 3    /* solvePnPRansac found no pose (:352) */
#define B200VO_LOOP_OVERFLOW 4      /* an append would exceed a capacity (landmarks, candidates or pose history) */
#define B200VO_LOOP_DETECT_LIMIT 5  /* more corner candidates in the frame than the batched detector ranks */
#define B200VO_LOOP_NO_BOOTSTRAP 6  /* the bootstrap found no essential matrix (fewer than 5 ratio-test matches, or RANSAC found no model) */

int b200vo_loop_create(b200vo_ctx* ctx, int batch, const b200vo_loop_cfg* cfg, b200vo_loop** out);
void b200vo_loop_destroy(b200vo_loop* lp);
/* Per-sequence camera intrinsics of the loop, as b200vo_batch_set_intrinsics: b200vo_loop_create gives every sequence
 * cfg->batch.K; afterwards sequence seqs[k] is tracked, posed, triangulated and bootstrapped with K[k] (double [n_seq][9]).
 * The state, status and frames of a sequence are not touched: a caller who hands a slot to another camera sets its K just
 * before b200vo_loop_load or b200vo_loop_bootstrap of that slot.  Same validation (B200VO_E_BADARG, nothing changes).
 * Synchronous. */
int b200vo_loop_set_intrinsics(b200vo_loop* lp, int n_seq, const int32_t* seqs, const double* K);
/* Per-sequence frame size of the loop, as b200vo_batch_set_frame_size (same validation: B200VO_E_BADARG, nothing changes).
 * The listed sequences become B200VO_LOOP_IDLE: their state arrays stay readable, and steps skip them until
 * b200vo_loop_load or b200vo_loop_bootstrap runs for them.  Their detection masks are cleared.  Synchronous. */
int b200vo_loop_set_frame_size(b200vo_loop* lp, int n_seq, const int32_t* seqs, const int32_t* rows, const int32_t* cols);
/* Per-sequence detection mask of the loop, as b200vo_batch_set_detection_mask (same layout and validation).  It applies to
 * the corners a step detects for feature adding and to both SIFT frames of b200vo_loop_bootstrap, so that a sequence's
 * results are those of the per-call masked forms on its frames; tracking, pose and triangulation do not read it.  The
 * state, status and frames are not touched.  Synchronous. */
int b200vo_loop_set_detection_mask(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* masks);
/* Per-sequence lens distortion of the loop, as b200vo_batch_set_distortion (same layout and validation: B200VO_E_BADARG,
 * nothing changes).  Every frame the loop takes (steps, submitted sets, b200vo_loop_load, both frames of
 * b200vo_loop_bootstrap) is raw camera output, undistorted on the device with the sequence's K before anything reads it;
 * the loaded state, keypoints, landmarks, poses, b200vo_loop_read_state and detection masks are in the undistorted image.
 * The listed sequences become B200VO_LOOP_IDLE until b200vo_loop_load or b200vo_loop_bootstrap runs for them.  Synchronous. */
int b200vo_loop_set_distortion(b200vo_loop* lp, int n_seq, const int32_t* seqs, const double* dist);
/* Per-sequence lens of the loop, as b200vo_batch_set_lens (same layout and validation: B200VO_E_BADARG, nothing changes).
 * Every frame the loop takes is undistorted into the camera K of the sequence; b200vo_loop_set_intrinsics keeps an
 * explicit raw camera.  The listed sequences become B200VO_LOOP_IDLE until b200vo_loop_load or b200vo_loop_bootstrap runs
 * for them.  Synchronous. */
int b200vo_loop_set_lens(b200vo_loop* lp, int n_seq, const int32_t* seqs, const int32_t* model, const double* coeffs,
                         const double* raw_K);
/* State of sequence `seq` after its bootstrap (host arrays): frame uint8 (rows,cols) tight at the sequence's own frame size
 * (b200vo_loop_set_frame_size) = the current frame;
 * lm float32 (n_lm,3) + lm_kp float32 (n_lm,2); keys / first_keys float32 (n_cand,2) + first_pose int32 (n_cand)
 * = potential_keys / potential_first_keys / potential_transforms; poses double (n_poses,12) = self.transforms as
 * (R_CW row-major | t_CW).  The sequence's status becomes B200VO_LOOP_OK.  Synchronous. */
int b200vo_loop_load(b200vo_loop* lp, int seq, const uint8_t* frame, const float* lm, const float* lm_kp, int n_lm,
                     const float* keys, const float* first_keys, const int32_t* first_pose, int n_cand,
                     const double* poses, int n_poses);
/* The reference's bootstrap (`initialization`, :209-245 and :295-330) for the n_seq distinct sequences seqs[], on the device:
 * SIFT on both frames, kNN(k=2) + ratio test (m.distance < ratio * n.distance), findEssentialMat(RANSAC, prob 0.99,
 * threshold 1.0, maxIters 1000), recoverPose (distanceThresh 50) on the inliers, t * sign(t_z), triangulation of the inliers
 * against [I | 0].  frames0 / frames1: uint8 [n_seq][rows][cols] host arrays (page-locked or pageable); frames1[k] becomes
 * sequence seqs[k]'s current frame.  On success the sequence holds exactly what b200vo_loop_load would give it from that
 * result (two poses) and its status is B200VO_LOOP_OK.  Per listed sequence: status (OK, NO_BOOTSTRAP or OVERFLOW: the
 * landmarks exceed max_landmarks or the too_short_baseline candidates max_candidates), num_pts = the essential-matrix
 * inlier count (0 for NO_BOOTSTRAP), n_lm / n_cand = the loaded counts (0 unless OK).  A sequence that fails keeps its
 * state arrays, takes the status and is skipped by steps until it is loaded or bootstrapped again.  Sequences not listed
 * are untouched.  Bad indices (out of range, repeated), n_seq < 1 or null arrays: B200VO_E_BADARG before any device work.
 * A sequence whose RANSAC subset draw exhausts the fixed table of cv2 random numbers also gets NO_BOOTSTRAP.
 * frames0 / frames1 keep the slot layout whatever the sequences' own frame sizes.
 * Synchronous; synchronises the host twice per SIFT chunk of frames of each distinct frame size among the listed sequences
 * plus three times, and once more per workspace that has to grow. */
int b200vo_loop_bootstrap(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames0, const uint8_t* frames1,
                          double ratio, int32_t* status, int32_t* num_pts, int32_t* n_lm, int32_t* n_cand);
/* The same arrays back (capacity-sized outputs: max_landmarks, max_candidates, max_frames rows), plus the counts and
 * the status.  Synchronous. */
int b200vo_loop_read_state(b200vo_loop* lp, int seq, float* lm, float* lm_kp, int32_t* n_lm, float* keys, float* first_keys,
                           int32_t* first_pose, int32_t* n_cand, double* poses, int32_t* n_poses, int32_t* status);
/* Frames of a future step, as b200vo_batch_submit_frames(_dev). */
int b200vo_loop_submit_frames(b200vo_loop* lp, const uint8_t* frames);
int b200vo_loop_submit_frames_dev(b200vo_loop* lp, const uint8_t* frames_dev);
/* One frame for every sequence (frames: batch x rows x cols uint8; NULL: the oldest submitted set).
 * Per sequence: status int32, n_inliers int32, n_lm int32, n_cand int32 after the step, pose_cw double (batch,12) =
 * the pose appended this step.  n_inliers and pose_cw are 0 unless status is B200VO_LOOP_OK.
 * One upload (the frames, unless submitted) and one read-back of the packed result block. */
int b200vo_loop_step(b200vo_loop* lp, const uint8_t* frames, int32_t* status, int32_t* n_inliers, int32_t* n_lm,
                     int32_t* n_cand, double* pose_cw);
/* The same with device pointers; asynchronous on the ctx stream (never synchronises the host). */
int b200vo_loop_step_dev(b200vo_loop* lp, const uint8_t* frames_dev, int32_t* status_dev, int32_t* n_inliers_dev,
                         int32_t* n_lm_dev, int32_t* n_cand_dev, double* pose_cw_dev);
/* Listed steps: a step that advances only the n_seq distinct sequences seqs[] (any order), for streams that do not tick
 * together (different lengths or frame rates, dropped frames).  frames: uint8 [n_seq][rows][cols] in the slot layout and
 * in list order (only these are uploaded); NULL: the oldest submitted set, which must have been submitted with the same
 * list by b200vo_loop_submit_frames_seqs(_dev).  Full and listed sets may alternate in the FIFO and are consumed in order;
 * b200vo_loop_step(NULL) refuses a listed set and a listed step a full one.
 * A listed sequence runs exactly the step it runs in a batch of one, bit for bit (nothing in a step depends on how many
 * steps the batch has taken), so its results and state depend only on its own frames and the calls that list it.  A
 * sequence that is not listed is not touched: its state, status and current frame stay as they are, and its next listed
 * step tracks from that frame.  A listed sequence that is not B200VO_LOOP_OK is reported as b200vo_loop_step reports it.
 * Results: n_seq rows in list order (status, n_inliers, n_lm, n_cand int32 [n_seq], pose_cw double [n_seq][12]).
 * seqs is a HOST array in all four calls, the _dev forms included: the call validates it and sizes its launches from
 * it; the library keeps its own copy, so the caller may reuse it as soon as the call returns.
 * B200VO_E_BADARG, before any device work and with nothing changed: n_seq < 1 or > batch, an index out of range or
 * repeated, a null array, frames == NULL with nothing submitted or with a set submitted with another list (or with none),
 * frames passed while submitted sets are waiting.
 * b200vo_loop_step_seqs synchronises as b200vo_loop_step (one upload of the listed frames, one read-back of n_seq rows);
 * the _dev forms never synchronise the host.  The pyramids, the detector and the loop kernels work for the listed
 * sequences only, the trackers and the pose chain see a count of 0 for the others, and every other sequence's current
 * pyramid is copied into the step's pyramid set. */
int b200vo_loop_step_seqs(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames, int32_t* status,
                          int32_t* n_inliers, int32_t* n_lm, int32_t* n_cand, double* pose_cw);
int b200vo_loop_step_seqs_dev(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames_dev, int32_t* status_dev,
                              int32_t* n_inliers_dev, int32_t* n_lm_dev, int32_t* n_cand_dev, double* pose_cw_dev);
/* Frames of a future listed step: uint8 [n_seq][rows][cols] (page-locked host memory, or device memory for _dev) for
 * the sequences seqs[] (host array), as b200vo_loop_submit_frames(_dev).  Same list validation. */
int b200vo_loop_submit_frames_seqs(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames);
int b200vo_loop_submit_frames_seqs_dev(b200vo_loop* lp, int n_seq, const int32_t* seqs, const uint8_t* frames_dev);

int b200vo_sync(b200vo_ctx* ctx);
/* Page-locked host memory for frame buffers: b200vo_batch_step DMAs straight out of such a
 * buffer (pageable memory is staged through an internal pinned copy first). */
void* b200vo_host_alloc(b200vo_ctx* ctx, size_t bytes);
void b200vo_host_free(b200vo_ctx* ctx, void* p);
/* Raw stream handle (cudaStream_t) so callers can record CUDA events on the launching stream. */
void* b200vo_stream(b200vo_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
