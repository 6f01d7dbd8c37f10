"""The lens maps whose undistorted camera Knew may differ from the raw camera K, as the test-only C oracle restates them
(oracle/lens_oracle.c): cv2.fisheye.undistortImage and cv2.undistort(..., newCameraMatrix=Knew), plus the fisheye lenses
and new cameras the lens tests share."""
import ctypes as C

import numpy as np

import oracle
import undistort_reference as U


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def _f64(a, n):
    return np.ascontiguousarray(np.asarray(a, np.float64).reshape(n))


def fisheye_map(K, D, Knew, rows, cols):
    """cv2.fisheye.initUndistortRectifyMap(K, D, I, Knew, (cols, rows), CV_16SC2) -> (xy int16 (rows, cols, 2), fr uint16)"""
    xy = np.empty((rows, cols, 2), np.int16)
    fr = np.empty((rows, cols), np.uint16)
    oracle.lib().orc_fisheye_map(rows, cols, _p(_f64(K, 9), C.c_double), _p(_f64(D, 4), C.c_double), _p(_f64(Knew, 9), C.c_double),
                                 _p(xy, C.c_int16), _p(fr, C.c_uint16))
    return xy, fr


def fisheye_source_px(K, D, Knew, rows, cols):
    """the source pixel (iu >> 5, iv >> 5) of every entry of the fisheye map before it is stored as int16, restated in
    numpy: int64 (rows, cols, 2).  fisheye_map holds it modulo 2^16."""
    K, Knew, D = np.asarray(K, np.float64), np.asarray(Knew, np.float64), np.asarray(D, np.float64)
    j, i = np.meshgrid(np.arange(cols, dtype=np.float64), np.arange(rows, dtype=np.float64))
    x, y = (j - Knew[0, 2]) / Knew[0, 0], (i - Knew[1, 2]) / Knew[1, 1]
    r = np.sqrt(x * x + y * y)
    th = np.arctan(r)
    th2 = th * th
    th4 = th2 * th2
    thd = th * (1 + D[0] * th2 + D[1] * th4 + D[2] * (th4 * th2) + D[3] * (th4 * th4))
    s = np.where(r == 0, 1.0, thd / np.where(r == 0, 1.0, r))
    iu = np.rint((K[0, 0] * x * s + K[0, 2]) * 32).astype(np.int64)
    iv = np.rint((K[1, 1] * y * s + K[1, 2]) * 32).astype(np.int64)
    return np.stack([iu >> 5, iv >> 5], -1)


def undistort_map_new(K, dist, Knew, rows, cols):
    """cv2.initUndistortRectifyMap(K, dist, None, Knew, (cols, rows), CV_16SC2) -> (xy, fr)"""
    xy = np.empty((rows, cols, 2), np.int16)
    fr = np.empty((rows, cols), np.uint16)
    oracle.lib().orc_undistort_map_new_camera(rows, cols, _p(_f64(K, 9), C.c_double), _p(_f64(U.dist8(dist), 8), C.c_double),
                                              _p(_f64(Knew, 9), C.c_double), _p(xy, C.c_int16), _p(fr, C.c_uint16))
    return xy, fr


def remap(img, xy, fr):
    img = np.ascontiguousarray(img, np.uint8)
    rows, cols = img.shape
    out = np.empty_like(img)
    oracle.lib().orc_remap_linear(_p(img, C.c_uint8), rows, cols, _p(np.ascontiguousarray(xy), C.c_int16),
                                  _p(np.ascontiguousarray(fr), C.c_uint16), _p(out, C.c_uint8))
    return out


def fisheye_undistort(img, K, D, Knew=None):
    """cv2.fisheye.undistortImage(img, K, D, Knew=Knew); Knew None is the identity, as in cv2"""
    return remap(img, *fisheye_map(K, D, np.eye(3) if Knew is None else Knew, *img.shape))


def undistort_new(img, K, dist, Knew):
    """cv2.undistort(img, K, dist, newCameraMatrix=Knew)"""
    return remap(img, *undistort_map_new(K, dist, Knew, *img.shape))


# fisheye cameras (K, D, rows, cols): a T265-like tracking camera, a wide VGA lens and a KITTI-sized one
K_T265 = np.array([[285.7, 0.0, 418.6], [0.0, 286.3, 405.2], [0.0, 0.0, 1.0]])
FISHEYE = {
    "t265": (K_T265, [-0.0070, 0.0437, -0.0410, 0.0076], 800, 848),
    "vga": (np.array([[320.0, 0.0, 319.5], [0.0, 321.0, 239.5], [0.0, 0.0, 1.0]]), [0.05, -0.02, 0.004, -0.0005], 480, 640),
    "kitti": (np.array([[420.0, 0.0, 620.3], [0.0, 418.0, 187.7], [0.0, 0.0, 1.0]]), [0.02, 0.01, -0.003, 0.0002], 376, 1241),
}
BALANCES = [0.0, 0.3, 0.7, 1.0]


def fisheye_knew(cv2, K, D, rows, cols, balance):
    """the undistorted camera a cv2 user picks for a fisheye lens"""
    return cv2.fisheye.estimateNewCameraMatrixForUndistortRectify(np.asarray(K, np.float64), np.asarray(D, np.float64).reshape(4, 1),
                                                                  (cols, rows), np.eye(3), balance=balance)


def pinhole_knew(cv2, K, dist, rows, cols, alpha):
    """cv2.getOptimalNewCameraMatrix(K, dist, size, alpha) (the full new camera, valid region ignored)"""
    return cv2.getOptimalNewCameraMatrix(np.asarray(K, np.float64), np.asarray(dist, np.float64), (cols, rows), alpha)[0]
