"""The masked-detection reference (tests/mask_reference.py) against live cv2 4.13: goodFeaturesToTrack(..., mask=) ordered
lists exact, SIFT detectAndCompute(img, mask) as the unmasked comparison of test_oracle_sift.py, and cv2's own masked
SIFT equal to its unmasked list filtered by the pixel rule."""
import numpy as np
import pytest

import mask_reference as R
import oracle
from monocular_visual_odometry_va4mr_b200 import synth
from sift_compare import compare

cv2 = pytest.importorskip("cv2")

GFTT_ARGS = (1400, 0.1, 10)     # the reference's feature options (main.py:28-33)


def _cv2_gftt(img, mask, mc=GFTT_ARGS[0], q=GFTT_ARGS[1], md=GFTT_ARGS[2]):
    return cv2.goodFeaturesToTrack(img, mc, q, md, mask=mask, blockSize=3)


def _same(a, b):
    if a is None or b is None:
        return a is None and b is None
    return a.shape == b.shape and np.array_equal(a, b)


@pytest.fixture(scope="module")
def frames():
    return [synth.render_sequence("kitti", 1, seed=s)["frames"][0] for s in (0, 7)]


def test_unmasked_reference_is_the_oracle(frames):
    for img in frames:
        assert _same(R.good_features_to_track(img, *GFTT_ARGS), oracle.good_features_to_track(img, *GFTT_ARGS, 3))


@pytest.mark.parametrize("name", ["hood", "wedges", "blobs", "all_255", "all_1", "all_7", "all_0", "quiet_patch", "patch_and_ring"])
def test_gftt_masks_on_rendered_frames(frames, name):
    for k, img in enumerate(frames):
        mask = R.standard_masks(img, seed=k)[name]
        want = _cv2_gftt(img, mask)
        assert _same(R.good_features_to_track(img, *GFTT_ARGS, mask=mask), want), (k, name)
        if name == "all_0":
            assert want is None
        if name in ("all_255", "all_1", "all_7"):
            assert _same(want, _cv2_gftt(img, None))


def test_gftt_mask_cases_that_move_the_threshold(frames):
    """A quiet patch's own maximum is far below the frame's, so it keeps corners an unmasked call drops; with the border
    ring in the mask the ring's stronger maximum sets the threshold again."""
    img = frames[0]
    eig = oracle.min_eig_map(img)
    m = R.patch_masks(img)
    patch, ring = m["quiet_patch"] != 0, m["patch_and_ring"] != 0
    assert eig[patch].max() < 0.05 * eig.max()
    assert eig[ring].max() > 2 * eig[patch].max()
    alone = _cv2_gftt(img, m["quiet_patch"])
    with_ring = _cv2_gftt(img, m["patch_and_ring"])
    unmasked = _cv2_gftt(img, None).reshape(-1, 2)
    inside = patch[unmasked[:, 1].astype(int), unmasked[:, 0].astype(int)].sum()
    assert alone is not None and len(alone) > inside
    assert with_ring is None or len(with_ring) < len(alone)


def test_gftt_one_pixel_mask_on_a_corner(frames):
    img = frames[0]
    for x, y in _cv2_gftt(img, None).reshape(-1, 2)[:5].astype(int):
        one = np.zeros(img.shape, np.uint8)
        one[y, x] = 1
        want = _cv2_gftt(img, one)
        assert want is not None and np.array_equal(want.reshape(-1, 2), [[x, y]])
        assert _same(R.good_features_to_track(img, *GFTT_ARGS, mask=one), want)


def test_gftt_negative_eigenvalue_masks():
    """Masks on pixels of negative eigenvalue (masked maximum < 0): cv2 finds nothing, and so does the reference."""
    cases = R.negative_eig_cases()
    assert len(cases) >= 3
    for img, one, nine in cases:
        eig = oracle.min_eig_map(img)
        assert eig[one != 0].max() < 0 and eig[nine != 0].max() < 0
        for m in (one, nine):
            for q in (0.01, 0.1, 1.0):
                want = cv2.goodFeaturesToTrack(img, 10, q, 1, mask=m)
                assert want is None
                assert R.good_features_to_track(img, 10, q, 1, mask=m) is None


@pytest.mark.parametrize("name", ["hood", "wedges", "blobs", "all_255", "all_1", "all_0", "quiet_patch", "patch_and_ring"])
def test_gftt_masks_on_the_checkerboard(name):
    """More than 32768 masked candidates for the large masks: the detector's bitonic sort path."""
    img = R.checkerboard()
    mask = R.standard_masks(img)[name]
    idx, _ = R.gftt_candidates(img, 0.5, mask)
    if name in ("hood", "wedges", "all_255", "all_1"):
        assert len(idx) > 32768
    want = cv2.goodFeaturesToTrack(img, 0, 0.5, 0, mask=mask)
    assert _same(R.good_features_to_track(img, 0, 0.5, 0, mask=mask), want)


def test_gftt_bad_masks_raise_in_cv2():
    img = np.zeros((60, 80), np.uint8)
    for bad in (np.zeros((10, 10), np.uint8), np.zeros((60, 80), np.float32), np.zeros((60, 80, 1), np.uint16)):
        with pytest.raises(cv2.error):
            cv2.goodFeaturesToTrack(img, 10, 0.1, 5, mask=bad)


def _cv2_sift(img, mask):
    kps, desc = cv2.SIFT_create().detectAndCompute(img, mask)
    kp = np.float32([[k.pt[0], k.pt[1], k.size, k.angle, k.response] for k in kps]).reshape(-1, 5)
    octv = np.int32([k.octave for k in kps])
    return kp, octv, (np.zeros((0, 128), np.float32) if desc is None else desc)


def _sift_masks(img, kp):
    """name -> mask: the standard ones, and one whose zero pixels sit where keypoints closest to x.5 / y.5 round to"""
    out = {k: v for k, v in R.standard_masks(img).items() if k in ("hood", "wedges", "blobs", "all_7", "all_0")}
    frac = np.abs(np.c_[kp[:, 0], kp[:, 1]] % 1 - 0.5).min(axis=1)
    m = np.full(img.shape, 255, np.uint8)
    for x, y in kp[np.argsort(frac)[:40], :2]:
        m[int(np.float32(y) + np.float32(0.5)), int(np.float32(x) + np.float32(0.5))] = 0
    out["half_pixel_edges"] = m
    return out


@pytest.mark.parametrize("seed", [0, 3])
def test_sift_mask_is_a_pixel_filter_in_cv2(seed):
    """cv2's masked list is its unmasked list filtered by the rounded-position rule: same order, fields and descriptors."""
    img = synth.render_sequence("kitti", 1, seed=seed, width=640, height=240)["frames"][0]
    kp0, oc0, d0 = _cv2_sift(img, None)
    for name, mask in _sift_masks(img, kp0).items():
        kp1, oc1, d1 = _cv2_sift(img, mask)
        keep = R.sift_mask_keep(kp0[:, :2], mask)
        assert np.array_equal(kp1, kp0[keep]) and np.array_equal(oc1, oc0[keep]) and np.array_equal(d1, d0[keep]), name
        if name == "half_pixel_edges":
            assert 0 < (~keep).sum() <= 40


@pytest.mark.parametrize("seed", [0, 3])
def test_sift_masked_reference_vs_cv2(seed):
    img = synth.render_sequence("kitti", 1, seed=seed, width=640, height=240)["frames"][0]
    kp0, _, _ = _cv2_sift(img, None)
    for name, mask in _sift_masks(img, kp0).items():
        kp, octv, desc = R.sift_detect_and_compute(img, mask)
        ckp, coct, cdesc = _cv2_sift(img, mask)
        compare(kp, octv, desc, ckp, coct, cdesc)
        if len(kp) == len(ckp):
            assert np.array_equal(octv, coct) and np.array_equal(kp[:, :2], ckp[:, :2]), name
