"""cv2.undistort(src, K, dist) (newCameraMatrix = K) as the test-only C oracle restates it (oracle/undistort_oracle.c): the
fixed-point map of initUndistortRectifyMap(..., CV_16SC2) and the bilinear BORDER_CONSTANT remap through it, plus the
distortion models and scenes the undistortion tests share."""
import ctypes as C

import numpy as np

import oracle
from monocular_visual_odometry_va4mr_b200 import synth


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def dist8(dist):
    """4, 5 or 8 coefficients (or None) -> the 8 of the oracle and of set_distortion"""
    d = np.zeros(8)
    if dist is not None:
        d[:len(dist)] = dist
    return d


def undistort_map(K, dist, rows, cols):
    """-> (xy int16 (rows, cols, 2), fr uint16 (rows, cols)) in cv2's CV_16SC2 + CV_16UC1 layout"""
    K = np.ascontiguousarray(K, np.float64).reshape(9)
    d = np.ascontiguousarray(dist8(dist))
    xy = np.empty((rows, cols, 2), np.int16)
    fr = np.empty((rows, cols), np.uint16)
    oracle.lib().orc_undistort_map(rows, cols, _p(K, C.c_double), _p(d, C.c_double), _p(xy, C.c_int16), _p(fr, C.c_uint16))
    return xy, fr


def undistort(img, K, dist):
    img = np.ascontiguousarray(img, np.uint8)
    rows, cols = img.shape
    xy, fr = undistort_map(K, dist, rows, cols)
    out = np.empty_like(img)
    oracle.lib().orc_remap_linear(_p(img, C.c_uint8), rows, cols, _p(xy, C.c_int16), _p(fr, C.c_uint16), _p(out, C.c_uint8))
    return out


# distortion models: name -> coefficients (4, 5 or 8)
MODELS = {
    "kitti_like_5": [-0.28, 0.07, 0.0002, 0.0001, -0.006],
    "plumb_4": [0.1, -0.05, 0.001, 0.002],
    "barrel_strong_5": [-0.45, 0.22, 0.0, 0.0, -0.06],
    "pincushion_5": [0.5, 0.3, 0.0, 0.0, 0.2],
    "rational_8": [0.3, 0.1, 0.001, -0.001, 0.0, -0.9, 0.1, 0.05],
    "rational_pole_8": [0.5, 0.0, 0.0, 0.0, 0.0, -3.0, 0.0, 0.0],   # the denominator changes sign inside the frame
    "zero_5": [0.0, 0.0, 0.0, 0.0, 0.0],
}

# the reference cameras at their frame sizes
CAMERAS = {"kitti": (synth.K_KITTI, 376, 1241), "malaga": (synth.K_MALAGA, 768, 1024), "parking": (synth.K_PARKING, 480, 640)}


def scale_K(K, rows, cols, rows0, cols0, frac=(0.0, 0.0)):
    """K of a camera of size rows0 x cols0 scaled to rows x cols, with (fx, fy) fractional offsets added to cx, cy"""
    K = np.array(K, np.float64)
    K[0] *= cols / cols0
    K[1] *= rows / rows0
    K[2, 2] = 1.0
    K[0, 2] += frac[0]
    K[1, 2] += frac[1]
    return K
