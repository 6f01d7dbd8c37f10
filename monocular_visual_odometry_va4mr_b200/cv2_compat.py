"""Drop-in replacements for the cv2 call sites on the reference's hot path.

Mirrors, argument for argument, the five ``cv2`` names used by the reference's
``VisualOdometryPipeLine.py``:

===============================  ==========================
``cv2.calcOpticalFlowPyrLK``     ``:281``, ``:287``
``cv2.goodFeaturesToTrack``      ``:256``
``cv2.BFMatcher().knnMatch``     ``:36``, ``:229`` (+ ratio loop ``:218-224``)
``cv2.findEssentialMat``         ``:308``
``cv2.solvePnPRansac``           ``:343``
===============================  ==========================

Same argument order, defaults, array shapes and dtypes, status / inlier-index layouts.
Everything runs on the B200 through ``libb200vo.so``; argument patterns the reference never
uses raise ``NotImplementedError`` -- never a silent CPU fallback.  ``install()`` patches the
names onto the real ``cv2`` module so the *unmodified* reference class picks them up.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import c_f32p, c_f64p, c_i32p, c_u8p

try:  # the reference imports cv2 for everything that is *not* on the hot path
    import cv2 as _cv2
    error = _cv2.error
except Exception:  # pragma: no cover - cv2-less box
    _cv2 = None

    class error(Exception):  # noqa: N801 - cv2 spells it lower-case
        pass

# cv2 constants used by the call sites
TERM_CRITERIA_COUNT = 1
TERM_CRITERIA_MAX_ITER = 1
TERM_CRITERIA_EPS = 2
RANSAC = 8
LMEDS = 4
SOLVEPNP_ITERATIVE = 0
SOLVEPNP_EPNP = 1
SOLVEPNP_P3P = 2
NORM_L2 = 4


def _ctx(device=None) -> _lib.Context:
    return _lib.default_context(0 if device is None else device)


def _raise(ctx: _lib.Context, rc: int, what: str):
    msg = ctx.last_error()
    if rc == -2:
        raise NotImplementedError(f"{what}: {msg} (b200vo implements only the reference's argument patterns; no CPU fallback)")
    if rc < 0:
        raise error(f"b200vo {what}: (-215:Assertion failed) {msg}")
    raise _lib.B200VOError(f"b200vo {what}: CUDA failure {rc}: {msg}")


def _p(a, t):
    return a.ctypes.data_as(t)


def _image_arg(img, name):
    if not isinstance(img, np.ndarray) or img.ndim != 2 or img.dtype != np.uint8:
        raise error(f"b200vo: {name} must be a 2-D uint8 array (the reference passes cv2.IMREAD_GRAYSCALE frames)")
    if img.strides[1] != 1 or img.strides[0] < img.shape[1]:
        img = np.ascontiguousarray(img)
    return img, img.strides[0]


# --------------------------------------------------------------------------------------
# cv2.calcOpticalFlowPyrLK  (reference :281, :287)
# --------------------------------------------------------------------------------------
_klt_cache = {"mode": "strict", "frames": {}}


def set_frame_cache(mode: str = "strict"):
    """``"strict"`` (default): every call uploads both images, as cv2 rebuilds both pyramids.
    ``"identity"``: device pyramids are reused when the *same ndarray object* is passed again
    (the reference passes ``self.potential_frame`` twice per frame and as ``prev`` of the next
    frame, ``:281,:287,:373``).  The shim holds a reference to the array, so ids stay unique;
    callers must not mutate a frame in place while it is cached (the reference never does)."""
    if mode not in ("strict", "identity"):
        raise ValueError(mode)
    _klt_cache["mode"] = mode
    _klt_cache["frames"].clear()


def _slot_for(ctx, img, step, win, max_level, tick):
    """identity cache: returns the device slot holding img's pyramid (uploading if needed)."""
    frames = _klt_cache["frames"]
    key = id(img)
    ent = frames.get(key)
    if ent is not None and ent["img"] is img and ent["win"] == win and ent["ml"] == max_level:
        ent["tick"] = tick
        return ent["slot"]
    used = {e["slot"] for e in frames.values()}
    free = [s for s in range(4) if s not in used]
    if free:
        slot = free[0]
    else:
        old = min(frames, key=lambda k: frames[k]["tick"])
        slot = frames.pop(old)["slot"]
    rc = ctx.lib.b200vo_frame_upload(ctx.h, slot, _p(img, c_u8p), img.shape[0], img.shape[1], step,
                                     win[0], win[1], max_level)
    if rc != 0:
        _raise(ctx, rc, "calcOpticalFlowPyrLK")
    frames[key] = dict(img=img, slot=slot, win=win, ml=max_level, tick=tick)
    return slot


_tick = [0]


def calcOpticalFlowPyrLK(prevImg, nextImg, prevPts, nextPts, status=None, err=None, winSize=(21, 21),
                         maxLevel=3, criteria=(TERM_CRITERIA_COUNT + TERM_CRITERIA_EPS, 30, 0.01),
                         flags=0, minEigThreshold=1e-4):
    """cv2.calcOpticalFlowPyrLK -> (nextPts, status, err); reference call sites :281, :287."""
    if nextPts is not None or status is not None or err is not None:
        raise NotImplementedError("b200vo calcOpticalFlowPyrLK: output/initial-flow arrays are not supported (the reference passes None)")
    prevImg, pstep = _image_arg(prevImg, "prevImg")
    nextImg, nstep = _image_arg(nextImg, "nextImg")
    if prevImg.shape != nextImg.shape:
        raise error("b200vo calcOpticalFlowPyrLK: (-215:Assertion failed) prevPyr[level * lvlStep1].size() == nextPyr[level * lvlStep2].size()")
    pts = np.asarray(prevPts)
    if pts.dtype != np.float32 or pts.ndim not in (2, 3) or pts.shape[-1] != 2 or (pts.ndim == 3 and 1 not in pts.shape[:2]):
        if pts.size == 0:
            return None, None, None
        raise error("b200vo calcOpticalFlowPyrLK: (-215:Assertion failed) (npoints = prevPtsMat.checkVector(2, CV_32F, true)) >= 0")
    n = pts.size // 2
    if n == 0:
        return None, None, None
    flat = np.ascontiguousarray(pts.reshape(n, 2))
    out = np.empty((n, 2), np.float32)
    st = np.empty((n, 1), np.uint8)
    er = np.empty((n, 1), np.float32)
    ctx = _ctx()
    win = (int(winSize[0]), int(winSize[1]))
    ctype, cmax, ceps = int(criteria[0]), int(criteria[1]), float(criteria[2])
    if _klt_cache["mode"] == "identity":
        _tick[0] += 1
        s_prev = _slot_for(ctx, prevImg, pstep, win, int(maxLevel), _tick[0])
        _tick[0] += 1
        s_next = _slot_for(ctx, nextImg, nstep, win, int(maxLevel), _tick[0])
        rc = ctx.lib.b200vo_klt_slots(ctx.h, s_prev, s_next, _p(flat, c_f32p), n, win[0], win[1], int(maxLevel),
                                      ctype, cmax, ceps, int(flags), float(minEigThreshold),
                                      _p(out, c_f32p), _p(st, c_u8p), _p(er, c_f32p))
    else:
        rc = ctx.lib.b200vo_calc_optical_flow_pyr_lk(
            ctx.h, _p(prevImg, c_u8p), _p(nextImg, c_u8p), prevImg.shape[0], prevImg.shape[1], pstep, nstep,
            _p(flat, c_f32p), n, win[0], win[1], int(maxLevel), ctype, cmax, ceps, int(flags),
            float(minEigThreshold), _p(out, c_f32p), _p(st, c_u8p), _p(er, c_f32p))
    if rc != 0:
        _raise(ctx, rc, "calcOpticalFlowPyrLK")
    return out.reshape(pts.shape), st, er


# --------------------------------------------------------------------------------------
# cv2.goodFeaturesToTrack  (reference :256)
# --------------------------------------------------------------------------------------
def goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, corners=None, mask=None, blockSize=3,
                        useHarrisDetector=False, k=0.04):
    """cv2.goodFeaturesToTrack -> float32 (M,1,2) or None; reference call site :256."""
    if mask is not None or useHarrisDetector or corners is not None:
        raise NotImplementedError("b200vo goodFeaturesToTrack: mask / Harris / preallocated corners are not supported")
    image, step = _image_arg(image, "image")
    if not (qualityLevel > 0 and minDistance >= 0 and maxCorners >= 0):
        raise error("b200vo goodFeaturesToTrack: (-215:Assertion failed) qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0")
    ctx = _ctx()
    cap = int(maxCorners) if maxCorners > 0 else image.shape[0] * image.shape[1]
    buf = np.empty((max(cap, 1), 2), np.float32)
    n_out = C.c_int(0)
    rc = ctx.lib.b200vo_good_features_to_track(ctx.h, _p(image, c_u8p), image.shape[0], image.shape[1], step,
                                               int(maxCorners), float(qualityLevel), float(minDistance),
                                               int(blockSize), _p(buf, c_f32p), C.byref(n_out))
    if rc != 0:
        _raise(ctx, rc, "goodFeaturesToTrack")
    if n_out.value == 0:
        return None
    return buf[:n_out.value].reshape(-1, 1, 2).copy()


def _mask_arg(mask, shape, what):
    """A detection mask: 2-D uint8 of the image's shape (cv2 raises cv2.error otherwise)."""
    if not isinstance(mask, np.ndarray) or mask.dtype != np.uint8 or mask.shape != shape:
        got = f"{mask.dtype} {mask.shape}" if isinstance(mask, np.ndarray) else type(mask).__name__
        raise error(f"b200vo {what}: (-215:Assertion failed) mask.empty() || (mask.type() == CV_8UC1 && mask.sameSize(image)): "
                    f"the mask must be uint8 {shape}, got {got}")
    return np.ascontiguousarray(mask)


def good_features_to_track_masked(image, maxCorners, qualityLevel, minDistance, mask, blockSize=3):
    """cv2.goodFeaturesToTrack(image, maxCorners, qualityLevel, minDistance, mask=mask, blockSize=blockSize) -> float32 (M,1,2)
    or None.  A corner needs a nonzero mask byte at its pixel, and the quality threshold is taken over the masked pixels
    only, as cv2 does.  mask=None: the unmasked call.  A mask that is not uint8 of the image's shape raises ``error``."""
    image, step = _image_arg(image, "image")
    if mask is not None:
        mask = _mask_arg(mask, image.shape, "goodFeaturesToTrack")
    if not (qualityLevel > 0 and minDistance >= 0 and maxCorners >= 0):
        raise error("b200vo goodFeaturesToTrack: (-215:Assertion failed) qualityLevel > 0 && minDistance >= 0 && maxCorners >= 0")
    ctx = _ctx()
    cap = int(maxCorners) if maxCorners > 0 else image.shape[0] * image.shape[1]
    buf = np.empty((max(cap, 1), 2), np.float32)
    n_out = C.c_int(0)
    rc = ctx.lib.b200vo_good_features_to_track_masked(ctx.h, _p(image, c_u8p), image.shape[0], image.shape[1], step,
                                                      None if mask is None else _p(mask, c_u8p), 0 if mask is None else mask.shape[1],
                                                      int(maxCorners), float(qualityLevel), float(minDistance), int(blockSize),
                                                      _p(buf, c_f32p), C.byref(n_out))
    if rc != 0:
        _raise(ctx, rc, "goodFeaturesToTrack")
    if n_out.value == 0:
        return None
    return buf[:n_out.value].reshape(-1, 1, 2).copy()


# --------------------------------------------------------------------------------------
# cv2.BFMatcher().knnMatch + ratio test  (reference :36, :229, :218-224)
# --------------------------------------------------------------------------------------
class DMatch:
    """Field-compatible with cv2.DMatch (the reference reads .distance/.queryIdx/.trainIdx)."""
    __slots__ = ("queryIdx", "trainIdx", "imgIdx", "distance")

    def __init__(self, queryIdx=-1, trainIdx=-1, distance=float("inf"), imgIdx=0):
        self.queryIdx, self.trainIdx, self.imgIdx, self.distance = queryIdx, trainIdx, imgIdx, distance

    def __repr__(self):
        return f"DMatch(q={self.queryIdx}, t={self.trainIdx}, d={self.distance})"


def knn2_ratio(queryDescriptors, trainDescriptors, ratio=0.8):
    """Fused array form: (idx int32 (Q,2), dist float32 (Q,2), accept uint8 (Q,)).

    idx/dist equal cv2.BFMatcher(NORM_L2).knnMatch(k=2); accept[i] equals the reference's
    ``m.distance < ratio * n.distance`` evaluated in float64 (``:221``)."""
    q = np.asarray(queryDescriptors)
    t = np.asarray(trainDescriptors)
    if q.ndim != 2 or t.ndim != 2 or q.shape[1] != t.shape[1] or q.dtype != np.float32 or t.dtype != np.float32:
        raise error("b200vo knnMatch: (-215:Assertion failed) type == src2.type() && src1.cols == src2.cols && (type == CV_32F || type == CV_8U)")
    q = np.ascontiguousarray(q)
    t = np.ascontiguousarray(t)
    nq, nt = q.shape[0], t.shape[0]
    idx = np.full((nq, 2), -1, np.int32)
    dist = np.full((nq, 2), np.finfo(np.float32).max, np.float32)
    acc = np.zeros((nq,), np.uint8)
    if nq == 0 or nt == 0:
        return idx, dist, acc
    ctx = _ctx()
    rc = ctx.lib.b200vo_knn2_ratio(ctx.h, _p(q, c_f32p), nq, _p(t, c_f32p), nt, q.shape[1], float(ratio),
                                   _p(idx, c_i32p), _p(dist, c_f32p), _p(acc, c_u8p))
    if rc != 0:
        _raise(ctx, rc, "knnMatch")
    return idx, dist, acc


class BFMatcher:
    """cv2.BFMatcher(normType=NORM_L2, crossCheck=False); only knnMatch(k<=2) is on the hot path."""

    def __init__(self, normType=NORM_L2, crossCheck=False):
        if normType != NORM_L2 or crossCheck:
            raise NotImplementedError("b200vo BFMatcher: only NORM_L2 without crossCheck (the reference's cv2.BFMatcher())")

    def knnMatch(self, queryDescriptors, trainDescriptors, k, mask=None, compactResult=False):
        if mask is not None or compactResult:
            raise NotImplementedError("b200vo knnMatch: mask/compactResult not supported")
        if k not in (1, 2):
            raise NotImplementedError("b200vo knnMatch: k must be 1 or 2 (the reference uses k=2)")
        idx, dist, _ = knn2_ratio(queryDescriptors, trainDescriptors, 0.8)
        out = []
        il = idx.tolist()
        dl = dist.astype(np.float64).tolist()
        for qi, (ii, dd) in enumerate(zip(il, dl)):
            row = [DMatch(qi, ii[j], dd[j]) for j in range(k) if ii[j] >= 0]
            out.append(tuple(row))
        return tuple(out)


# --------------------------------------------------------------------------------------
# cv2.SIFT_create().detectAndCompute  (reference :35, :226-227; SURVEY 8f row f4)
# --------------------------------------------------------------------------------------
class KeyPoint:
    """Field-compatible with cv2.KeyPoint (the reference reads .pt, :232-233)."""
    __slots__ = ("pt", "size", "angle", "response", "octave", "class_id")

    def __init__(self, x=0.0, y=0.0, size=0.0, angle=-1.0, response=0.0, octave=0, class_id=-1):
        self.pt, self.size, self.angle, self.response, self.octave, self.class_id = (x, y), size, angle, response, octave, class_id

    def __repr__(self):
        return f"KeyPoint(pt={self.pt}, size={self.size}, angle={self.angle}, octave={self.octave})"


def sift_detect_and_compute(image, max_keypoints=1 << 17, mask=None):
    """Array form: (kp float32 (n, 5) = x, y, size, angle, response; octave int32 (n,); descriptors float32 (n, 128)),
    rows in cv2's output order.  ``mask``: cv2's detectAndCompute(image, mask), uint8 of the image's shape; a keypoint is
    dropped where the byte at its rounded position is 0, the others keep their order and descriptors.  Unlike cv2, which
    does not check it, a mask of another shape or dtype raises ``error``."""
    img, step = _image_arg(image, "SIFT.detectAndCompute image")
    if mask is not None:
        mask = _mask_arg(mask, img.shape, "SIFT.detectAndCompute")
    ctx = _ctx()
    rows, cols = img.shape
    cap = 8192
    while True:
        kps = np.empty((cap, 6), np.float32)
        desc = np.empty((cap, 128), np.float32)
        n = C.c_int32(0)
        if mask is None:
            rc = ctx.lib.b200vo_sift_detect_and_compute(ctx.h, _p(img, c_u8p), rows, cols, step, cap, _p(kps, c_f32p), _p(desc, c_f32p),
                                                        C.byref(n))
        else:
            rc = ctx.lib.b200vo_sift_detect_and_compute_masked(ctx.h, _p(img, c_u8p), rows, cols, step, _p(mask, c_u8p), cols, cap,
                                                               _p(kps, c_f32p), _p(desc, c_f32p), C.byref(n))
        if rc != 0:
            _raise(ctx, rc, "SIFT.detectAndCompute")
        if n.value <= cap or cap >= max_keypoints:
            break
        cap = min(max_keypoints, max(n.value, 2 * cap))      # rare: more keypoints than the first buffer holds
    m = min(n.value, cap)
    return kps[:m, :5].copy(), kps[:m, 5].copy().view(np.int32), desc[:m].copy()


class SIFT:
    """cv2.SIFT_create() with the default parameters, as the reference constructs it (:35)."""

    def __init__(self, nfeatures=0, nOctaveLayers=3, contrastThreshold=0.04, edgeThreshold=10, sigma=1.6, enable_precise_upscale=False):
        if (nfeatures, nOctaveLayers, float(contrastThreshold), float(edgeThreshold), float(sigma), bool(enable_precise_upscale)) != (0, 3, 0.04, 10.0, 1.6, False):
            raise NotImplementedError("b200vo SIFT: only cv2.SIFT_create()'s default parameters (the reference's call)")

    def detectAndCompute(self, image, mask, descriptors=None, useProvidedKeypoints=False):
        if mask is not None or useProvidedKeypoints:
            raise NotImplementedError("b200vo SIFT.detectAndCompute: mask / useProvidedKeypoints are not supported (the reference passes None)")
        kp, octave, desc = sift_detect_and_compute(image)
        if _cv2 is not None:        # real cv2.KeyPoint objects when cv2 is there (drawKeypoints etc. keep working)
            kps = tuple(_cv2.KeyPoint(float(r[0]), float(r[1]), float(r[2]), float(r[3]), float(r[4]), int(o), -1) for r, o in zip(kp, octave))
        else:
            kps = tuple(KeyPoint(float(r[0]), float(r[1]), float(r[2]), float(r[3]), float(r[4]), int(o)) for r, o in zip(kp, octave))
        return kps, (desc if len(desc) else None)

    def descriptorSize(self):
        return 128

    def defaultNorm(self):
        return NORM_L2


def SIFT_create(*args, **kwargs):
    return SIFT(*args, **kwargs)


# --------------------------------------------------------------------------------------
# cv2.findEssentialMat  (reference :308)
# --------------------------------------------------------------------------------------
def findEssentialMat(points1, points2, cameraMatrix=None, method=RANSAC, prob=0.999, threshold=1.0,
                     maxIters=1000, mask=None):
    """cv2.findEssentialMat(points1, points2, K, method=RANSAC, prob=, threshold=) -> (E, mask)."""
    if method != RANSAC or mask is not None or cameraMatrix is None:
        raise NotImplementedError("b200vo findEssentialMat: only (points1, points2, K, method=RANSAC, prob, threshold[, maxIters])")
    p1 = np.ascontiguousarray(np.asarray(points1, np.float32).reshape(-1, 2))
    p2 = np.ascontiguousarray(np.asarray(points2, np.float32).reshape(-1, 2))
    if p1.shape != p2.shape:
        raise error("b200vo findEssentialMat: (-215:Assertion failed) npoints >= 0 && points2.checkVector(2) == npoints")
    n = p1.shape[0]
    if n < 5:
        return None, None
    K = np.ascontiguousarray(np.asarray(cameraMatrix, np.float64).reshape(3, 3))
    E = np.zeros((3, 3), np.float64)
    m = np.zeros((n, 1), np.uint8)
    found = C.c_int(0)
    ctx = _ctx()
    rc = ctx.lib.b200vo_find_essential_mat_ransac(ctx.h, _p(p1, c_f32p), _p(p2, c_f32p), n, _p(K, c_f64p), float(prob),
                                                  float(threshold), int(maxIters), _p(E, c_f64p), _p(m, c_u8p),
                                                  C.byref(found))
    if rc != 0:
        _raise(ctx, rc, "findEssentialMat")
    if not found.value:
        return None, None
    return E, m


# --------------------------------------------------------------------------------------
# cv2.recoverPose  (reference :315; SURVEY 8f row f3)
# --------------------------------------------------------------------------------------
def recoverPose(E, points1, points2, cameraMatrix=None, R=None, t=None, mask=None, distanceThresh=50.0):
    """cv2.recoverPose(E, points1, points2, K) -> (retval, R (3,3), t (3,1), mask (n,1) uint8 0/255)."""
    if cameraMatrix is None or R is not None or t is not None or mask is not None:
        raise NotImplementedError("b200vo recoverPose: only (E, points1, points2, cameraMatrix[, distanceThresh=]) (reference :315)")
    Em = np.ascontiguousarray(np.asarray(E, np.float64).reshape(3, 3))
    p1 = np.ascontiguousarray(np.asarray(points1, np.float32).reshape(-1, 2))
    p2 = np.ascontiguousarray(np.asarray(points2, np.float32).reshape(-1, 2))
    if p1.shape != p2.shape:
        raise error("b200vo recoverPose: (-215:Assertion failed) npoints >= 0 && points2.checkVector(2) == npoints")
    n = p1.shape[0]
    K = np.ascontiguousarray(np.asarray(cameraMatrix, np.float64).reshape(3, 3))
    Ro = np.zeros((3, 3), np.float64)
    to = np.zeros((3, 1), np.float64)
    m = np.zeros((n, 1), np.uint8)
    good = C.c_int(0)
    ctx = _ctx()
    rc = ctx.lib.b200vo_recover_pose(ctx.h, _p(Em, c_f64p), _p(p1, c_f32p), _p(p2, c_f32p), n, _p(K, c_f64p), float(distanceThresh),
                                     _p(Ro, c_f64p), _p(to, c_f64p), _p(m, c_u8p), C.byref(good))
    if rc != 0:
        _raise(ctx, rc, "recoverPose")
    return good.value, Ro, to, m


# --------------------------------------------------------------------------------------
# cv2.undistort and cv2.fisheye.undistortImage  (raw frames of cameras with lens distortion)
# --------------------------------------------------------------------------------------
def _pinhole_arg(M, name, what):
    """a 3 x 3 camera matrix argument: ``error`` unless 3 x 3, ``NotImplementedError`` unless a pinhole (no skew, last row
    0 0 1); its other checks (fx, fy > 0, finite) are the library's"""
    M = np.asarray(M, np.float64)
    if M.shape != (3, 3):
        raise error(f"b200vo {what}: (-215:Assertion failed) {name} is 3x3")
    if M[0, 1] != 0 or M[1, 0] != 0 or M[2, 0] != 0 or M[2, 1] != 0 or M[2, 2] != 1:
        raise NotImplementedError(f"b200vo {what}: only pinhole camera matrices (no skew, last row 0 0 1)")
    return np.ascontiguousarray(M)


def undistort(src, cameraMatrix, distCoeffs, dst=None, newCameraMatrix=None):
    """cv2.undistort(src, cameraMatrix, distCoeffs, newCameraMatrix=) -> uint8 image of src's shape, byte for byte what cv2
    computes.  src: 2-D uint8.  distCoeffs: 4, 5 or 8 coefficients (k1, k2, p1, p2[, k3[, k4, k5, k6]]) or None (a copy).
    newCameraMatrix: the pinhole camera of the undistorted image (e.g. from ``cv2.getOptimalNewCameraMatrix``), None:
    cameraMatrix.  Multi-channel images, the 12- and 14-coefficient models and camera matrices with skew or another last
    row raise ``NotImplementedError``; a bad camera matrix or non-finite coefficients raise ``error``."""
    if isinstance(src, np.ndarray) and src.ndim == 3:
        raise NotImplementedError("b200vo undistort: single-channel images only")
    src, step = _image_arg(src, "src")
    K = _pinhole_arg(cameraMatrix, "cameraMatrix", "undistort")
    Kn = K if newCameraMatrix is None else _pinhole_arg(newCameraMatrix, "newCameraMatrix", "undistort")
    d = np.zeros(4) if distCoeffs is None else np.asarray(distCoeffs, np.float64).reshape(-1)
    if d.size in (12, 14):
        raise NotImplementedError("b200vo undistort: the thin-prism (12) and tilted (14) models are not supported")
    if d.size not in (4, 5, 8):
        raise error("b200vo undistort: (-215:Assertion failed) distCoeffs has 4, 5, 8, 12 or 14 elements")
    d = np.ascontiguousarray(d)
    out = np.empty(src.shape, np.uint8)
    ctx = _ctx()
    rc = ctx.lib.b200vo_undistort_new_camera(ctx.h, _p(src, c_u8p), src.shape[0], src.shape[1], step, _p(K, c_f64p), _p(d, c_f64p),
                                             d.size, _p(Kn, c_f64p), _p(out, c_u8p))
    if rc != 0:
        _raise(ctx, rc, "undistort")
    if dst is not None:
        dst[...] = out
        return dst
    return out


def fisheye_undistort_image(distorted, K, D, undistorted=None, Knew=None, new_size=None):
    """cv2.fisheye.undistortImage(distorted, K, D, Knew=, new_size=) -> uint8 image of distorted's shape, byte for byte what
    cv2 computes.  distorted: 2-D uint8.  D: the 4 coefficients k1, k2, k3, k4.  Knew: the pinhole camera of the undistorted
    image (usually K, or ``cv2.fisheye.estimateNewCameraMatrixForUndistortRectify``'s); None is the identity, as in cv2.
    Multi-channel images, camera matrices with skew or another last row and a new_size other than the image's raise
    ``NotImplementedError``; a bad camera matrix, a D without 4 elements or non-finite coefficients raise ``error``."""
    if isinstance(distorted, np.ndarray) and distorted.ndim == 3:
        raise NotImplementedError("b200vo fisheye.undistortImage: single-channel images only")
    src, step = _image_arg(distorted, "distorted")
    K = _pinhole_arg(K, "K", "fisheye.undistortImage")
    Kn = None if Knew is None else _pinhole_arg(Knew, "Knew", "fisheye.undistortImage")
    if new_size is not None and tuple(new_size) not in ((0, 0), (src.shape[1], src.shape[0])):
        raise NotImplementedError("b200vo fisheye.undistortImage: new_size must be the image's (width, height)")
    d = np.ascontiguousarray(np.asarray(D, np.float64).reshape(-1))
    if d.size != 4:
        raise error("b200vo fisheye.undistortImage: (-215:Assertion failed) D.total() == 4")
    out = np.empty(src.shape, np.uint8)
    ctx = _ctx()
    rc = ctx.lib.b200vo_fisheye_undistort(ctx.h, _p(src, c_u8p), src.shape[0], src.shape[1], step, _p(K, c_f64p), _p(d, c_f64p),
                                          None if Kn is None else _p(Kn, c_f64p), _p(out, c_u8p))
    if rc != 0:
        _raise(ctx, rc, "fisheye.undistortImage")
    if undistorted is not None:
        undistorted[...] = out
        return undistorted
    return out


# --------------------------------------------------------------------------------------
# cv2.solvePnPRansac  (reference :343)
# --------------------------------------------------------------------------------------
def solvePnPRansac(objectPoints, imagePoints, cameraMatrix, distCoeffs, rvec=None, tvec=None,
                   useExtrinsicGuess=False, iterationsCount=100, reprojectionError=8.0, confidence=0.99,
                   inliers=None, flags=SOLVEPNP_ITERATIVE):
    """cv2.solvePnPRansac(..., flags=SOLVEPNP_P3P) -> (retval, rvec (3,1), tvec (3,1), inliers (M,1) int32 | None)."""
    if flags != SOLVEPNP_P3P or useExtrinsicGuess or rvec is not None or tvec is not None or inliers is not None:
        raise NotImplementedError("b200vo solvePnPRansac: only flags=SOLVEPNP_P3P without extrinsic guess (reference :343)")
    if distCoeffs is not None and np.any(np.asarray(distCoeffs) != 0):
        raise NotImplementedError("b200vo solvePnPRansac: non-zero distortion is not supported (the reference passes zeros(4))")
    obj = np.ascontiguousarray(np.asarray(objectPoints, np.float32).reshape(-1, 3))
    img = np.ascontiguousarray(np.asarray(imagePoints, np.float32).reshape(-1, 2))
    n = obj.shape[0]
    if n < 4 or img.shape[0] != n:
        raise error("b200vo solvePnPRansac: (-215:Assertion failed) npoints >= 4 && npoints == std::max(ipoints.checkVector(2, CV_32F), ipoints.checkVector(2, CV_64F))")
    K = np.ascontiguousarray(np.asarray(cameraMatrix, np.float64).reshape(3, 3))
    rv = np.zeros((3, 1), np.float64)
    tv = np.zeros((3, 1), np.float64)
    inl = np.empty((n,), np.int32)
    n_in = C.c_int(0)
    ok = C.c_int(0)
    ctx = _ctx()
    rc = ctx.lib.b200vo_solve_pnp_ransac_p3p(ctx.h, _p(obj, c_f32p), _p(img, c_f32p), n, _p(K, c_f64p),
                                             int(iterationsCount), float(reprojectionError), float(confidence),
                                             _p(rv, c_f64p), _p(tv, c_f64p), _p(inl, c_i32p), C.byref(n_in), C.byref(ok))
    if rc != 0:
        _raise(ctx, rc, "solvePnPRansac")
    if not ok.value:
        return False, rv, tv, None
    return True, rv, tv, inl[:n_in.value].reshape(-1, 1).copy()


# --------------------------------------------------------------------------------------
# installation onto the real cv2 module (route (i) of SURVEY.md 8b)
# --------------------------------------------------------------------------------------
_PATCHED = ("calcOpticalFlowPyrLK", "goodFeaturesToTrack", "BFMatcher", "findEssentialMat", "solvePnPRansac", "recoverPose", "SIFT_create")
_saved: dict = {}


def install(names=_PATCHED, cv2_module=None):
    """setattr the B200 implementations onto ``cv2`` so the unmodified reference class uses them."""
    mod = cv2_module or _cv2
    if mod is None:
        raise RuntimeError("cv2 is not importable; nothing to patch")
    for nm in names:
        if nm not in _saved:
            _saved[nm] = getattr(mod, nm)
        setattr(mod, nm, globals()[nm])
    return mod


def uninstall(cv2_module=None):
    mod = cv2_module or _cv2
    for nm, fn in list(_saved.items()):
        setattr(mod, nm, fn)
        del _saved[nm]


def __getattr__(name):
    """Anything that is not on the hot path (Rodrigues, triangulatePoints, ...) is the real cv2's."""
    if _cv2 is not None and hasattr(_cv2, name):
        return getattr(_cv2, name)
    raise AttributeError(name)
