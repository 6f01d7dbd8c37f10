"""The undistortion oracle (tests/undistort_reference.py) against live cv2 4.13: cv2.undistort byte for byte, and the map
against cv2.initUndistortRectifyMap(K, dist, None, K, size, CV_16SC2) bit for bit, on the reference cameras at their frame
sizes, 4-, 5- and 8-coefficient models, strong barrel and pincushion distortion, a rational model whose denominator changes
sign inside the frame, all-zero coefficients, small frames and principal points with fractional parts."""
import numpy as np
import pytest

import undistort_reference as U
from monocular_visual_odometry_va4mr_b200 import synth

cv2 = pytest.importorskip("cv2")


def _frame(rows, cols, seed):
    """a rendered frame of the requested size (scene texture, not noise: the remap's interpolation sees real gradients),
    with a few random bytes so that no region is flat"""
    f = synth.render_sequence("kitti", 1, seed=seed, width=max(cols, 64), height=max(rows, 48))["frames"][0][:rows, :cols].copy()
    rng = np.random.default_rng(seed)
    f[rng.random(f.shape) < 0.02] = rng.integers(0, 256, dtype=np.uint8)
    return f


def _check_map(K, dist, rows, cols):
    m1, m2 = cv2.initUndistortRectifyMap(K, np.asarray(dist, np.float64), None, K, (cols, rows), cv2.CV_16SC2)
    xy, fr = U.undistort_map(K, dist, rows, cols)
    # Entries whose source pixel saturates int16 lie far outside any image.  There cv2's order of double operations may
    # round the 1/32 px fraction differently (next to a pole of the rational model); both must saturate the same way.
    sat = (np.abs(m1.astype(np.int32)) >= 32767).any(-1)
    assert np.array_equal(sat, (np.abs(xy.astype(np.int32)) >= 32767).any(-1))
    assert np.array_equal(np.sign(m1[sat]), np.sign(xy[sat]))
    assert np.array_equal(m1[~sat], xy[~sat]) and np.array_equal(m2[~sat], fr[~sat])
    return int(sat.sum())


CASES = [(cam, model) for cam in U.CAMERAS for model in U.MODELS]


@pytest.mark.parametrize("cam,model", CASES)
def test_reference_cameras(cam, model):
    K, rows, cols = U.CAMERAS[cam]
    dist = U.MODELS[model]
    _check_map(K, dist, rows, cols)
    img = _frame(rows, cols, seed=len(model))
    ref = cv2.undistort(img, K, np.asarray(dist, np.float64))
    assert np.array_equal(U.undistort(img, K, dist), ref)
    if model == "zero_5":
        assert np.array_equal(ref, img)


def test_cases_cover_zero_regions_and_non_finite_values():
    K, rows, cols = U.CAMERAS["kitti"]
    img = np.full((rows, cols), 200, np.uint8)
    assert (U.undistort(img, K, U.MODELS["pincushion_5"]) == 0).sum() > 50000
    assert _check_map(K, U.MODELS["rational_pole_8"], rows, cols) > 0


@pytest.mark.parametrize("rows,cols", [(16, 16), (17, 23), (48, 64), (97, 131)])
@pytest.mark.parametrize("model", ["plumb_4", "barrel_strong_5", "pincushion_5", "rational_8"])
def test_small_frames(rows, cols, model):
    K, r0, c0 = U.CAMERAS["kitti"]
    K = U.scale_K(K, rows, cols, r0, c0)
    dist = U.MODELS[model]
    _check_map(K, dist, rows, cols)
    img = _frame(rows, cols, seed=rows * cols)
    assert np.array_equal(U.undistort(img, K, dist), cv2.undistort(img, K, np.asarray(dist, np.float64)))


@pytest.mark.parametrize("frac", [(0.5, 0.5), (0.3125, -0.71875), (0.1, 0.9), (-0.03125, 0.015625)])
@pytest.mark.parametrize("model", ["kitti_like_5", "rational_8"])
def test_fractional_principal_point(frac, model):
    K, rows, cols = U.CAMERAS["parking"]
    K = U.scale_K(K, rows, cols, rows, cols, frac)
    dist = U.MODELS[model]
    _check_map(K, dist, rows, cols)
    img = _frame(rows, cols, seed=3)
    assert np.array_equal(U.undistort(img, K, dist), cv2.undistort(img, K, np.asarray(dist, np.float64)))


def test_remap_through_cv2_map_is_undistort():
    K, rows, cols = U.CAMERAS["malaga"]
    dist = np.asarray(U.MODELS["barrel_strong_5"])
    img = _frame(rows, cols, seed=9)
    m1, m2 = cv2.initUndistortRectifyMap(K, dist, None, K, (cols, rows), cv2.CV_16SC2)
    assert np.array_equal(cv2.remap(img, m1, m2, cv2.INTER_LINEAR), U.undistort(img, K, dist))
