"""The lens oracle (tests/lens_reference.py) against live cv2 4.13: the fisheye map against
cv2.fisheye.initUndistortRectifyMap(K, D, I, Knew, size, CV_16SC2) and the pinhole new-camera map against
cv2.initUndistortRectifyMap(K, dist, None, Knew, size, CV_16SC2) bit for bit, and cv2.fisheye.undistortImage /
cv2.undistort(newCameraMatrix=) byte for byte.  Cases: fisheye cameras at their sizes with Knew = K and with
estimateNewCameraMatrixForUndistortRectify at four balances, a Knew whose map wraps int16, all-zero D, a principal point on
an integer pixel (r == 0), frames down to 16 x 16, fractional principal points, and 4-, 5- and 8-coefficient pinhole models
with getOptimalNewCameraMatrix at alpha 0, 0.5 and 1."""
import numpy as np
import pytest

import lens_reference as L
import undistort_reference as U
from monocular_visual_odometry_va4mr_b200 import synth

cv2 = pytest.importorskip("cv2")


def _frame(rows, cols, seed):
    """a rendered frame with a few random bytes (as in test_oracle_undistort.py)"""
    f = synth.render_sequence("kitti", 1, seed=seed, width=max(cols, 64), height=max(rows, 48))["frames"][0][:rows, :cols].copy()
    rng = np.random.default_rng(seed)
    f[rng.random(f.shape) < 0.02] = rng.integers(0, 256, dtype=np.uint8)
    return f


def _check_fisheye(K, D, Knew, rows, cols, seed=0):
    D = np.asarray(D, np.float64)
    m1, m2 = cv2.fisheye.initUndistortRectifyMap(K, D, np.eye(3), Knew, (cols, rows), cv2.CV_16SC2)
    xy, fr = L.fisheye_map(K, D, Knew, rows, cols)
    assert np.array_equal(m1, xy) and np.array_equal(m2, fr)
    img = _frame(rows, cols, seed)
    assert np.array_equal(L.fisheye_undistort(img, K, D, Knew), cv2.fisheye.undistortImage(img, K, D, Knew=Knew))
    return m1


def _check_pinhole(K, dist, Knew, rows, cols, seed=0):
    d = np.asarray(dist, np.float64)
    m1, m2 = cv2.initUndistortRectifyMap(K, d, None, Knew, (cols, rows), cv2.CV_16SC2)
    xy, fr = L.undistort_map_new(K, d, Knew, rows, cols)
    assert np.array_equal(m1, xy) and np.array_equal(m2, fr)
    img = _frame(rows, cols, seed)
    assert np.array_equal(L.undistort_new(img, K, d, Knew), cv2.undistort(img, K, d, newCameraMatrix=Knew))


@pytest.mark.parametrize("balance", [None] + L.BALANCES)
@pytest.mark.parametrize("cam", list(L.FISHEYE))
def test_fisheye_cameras(cam, balance):
    K, D, rows, cols = L.FISHEYE[cam]
    Knew = K if balance is None else L.fisheye_knew(cv2, K, D, rows, cols, balance)
    _check_fisheye(K, D, Knew, rows, cols, seed=rows)


def test_fisheye_identity_knew_is_cv2_default():
    K, D, rows, cols = L.FISHEYE["vga"]
    img = _frame(rows, cols, 4)
    assert np.array_equal(L.fisheye_undistort(img, K, D), cv2.fisheye.undistortImage(img, K, np.asarray(D, np.float64)))


def test_fisheye_map_wraps_int16():
    """a Knew with fx' ~ 0.001 takes theta to ~pi/2, where a strong lens sends the map far outside int16: cv2 stores
    (short)(iu >> 5), which wraps"""
    K, _, rows, cols = L.FISHEYE["t265"]
    D = np.array([0.5, 0.5, 1.0, 5.0])
    Knew = np.array([[0.001, 0.0, cols / 2], [0.0, 0.0012, rows / 2], [0.0, 0.0, 1.0]])
    m1 = _check_fisheye(K, D, Knew, rows, cols)
    src = L.fisheye_source_px(K, D, Knew, rows, cols)
    far = (np.abs(src) > 32767).any(-1)
    assert far.sum() > rows * cols // 4
    assert np.array_equal(m1[far], ((src[far] + 32768) % 65536 - 32768).astype(np.int16))


def test_fisheye_zero_coefficients_and_centre_pixel():
    """all-zero D is the equidistant projection (not the identity); cx, cy on an integer pixel hits r == 0"""
    K = np.array([[300.0, 0.0, 320.0], [0.0, 300.0, 240.0], [0.0, 0.0, 1.0]])
    m1 = _check_fisheye(K, [0, 0, 0, 0], K, 480, 640)
    assert tuple(m1[240, 320]) == (320, 240)
    ident = np.stack(np.meshgrid(np.arange(640), np.arange(480)), -1)
    assert (m1 != ident).any()
    _check_fisheye(K, L.FISHEYE["vga"][1], K, 480, 640)


@pytest.mark.parametrize("rows,cols", [(16, 16), (17, 23), (48, 64), (97, 131)])
@pytest.mark.parametrize("cam", ["t265", "kitti"])
def test_fisheye_small_frames(rows, cols, cam):
    K, D, r0, c0 = L.FISHEYE[cam]
    K = U.scale_K(K, rows, cols, r0, c0)
    _check_fisheye(K, D, K, rows, cols, seed=rows * cols)
    _check_fisheye(K, D, L.fisheye_knew(cv2, K, D, rows, cols, 0.5), rows, cols, seed=rows + cols)


@pytest.mark.parametrize("frac", [(0.5, 0.5), (0.3125, -0.71875), (0.1, 0.9), (-0.03125, 0.015625)])
def test_fisheye_fractional_principal_point(frac):
    K, D, rows, cols = L.FISHEYE["vga"]
    K = U.scale_K(K, rows, cols, rows, cols, frac)
    _check_fisheye(K, D, K, rows, cols, seed=3)
    _check_fisheye(K, D, L.fisheye_knew(cv2, K, D, rows, cols, 0.3), rows, cols, seed=5)


@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("model", ["plumb_4", "kitti_like_5", "barrel_strong_5", "rational_8"])
@pytest.mark.parametrize("cam", list(U.CAMERAS))
def test_pinhole_new_camera(cam, model, alpha):
    K, rows, cols = U.CAMERAS[cam]
    d = U.MODELS[model]
    _check_pinhole(K, d, L.pinhole_knew(cv2, K, d, rows, cols, alpha), rows, cols, seed=len(model))


@pytest.mark.parametrize("rows,cols", [(16, 16), (48, 64)])
def test_pinhole_new_camera_small_frames_and_fractional_point(rows, cols):
    K, r0, c0 = U.CAMERAS["parking"]
    K = U.scale_K(K, rows, cols, r0, c0, (0.3125, -0.71875))
    d = U.MODELS["barrel_strong_5"]
    for alpha in (0.0, 1.0):
        _check_pinhole(K, d, L.pinhole_knew(cv2, K, d, rows, cols, alpha), rows, cols, seed=rows)


def test_pinhole_new_camera_equal_to_K_is_the_old_map():
    K, rows, cols = U.CAMERAS["kitti"]
    d = U.MODELS["kitti_like_5"]
    xy, fr = L.undistort_map_new(K, d, K, rows, cols)
    xy0, fr0 = U.undistort_map(K, d, rows, cols)
    assert np.array_equal(xy, xy0) and np.array_equal(fr, fr0)
