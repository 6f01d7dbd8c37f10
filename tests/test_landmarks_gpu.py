"""CUDA versions of the two components next to the hot path (SURVEY.md 8f) through the C ABI: identical
masks and appended rows as the unmodified reference class produced (tests/golden/reference_trace.npz),
as the oracle, and as the reference's own numpy expression / live cv2.triangulatePoints."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from monocular_visual_odometry_va4mr_b200 import cv2_compat, hotpath

pytestmark = pytest.mark.gpu
OPT = lambda cfg: dict(min_dist_landmarks=cfg[0], max_dist_landmarks=cfg[1], min_baseline_angle=cfg[2], min_baseline_frames=int(cfg[3]))


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "reference_trace.npz"))


def test_min_distance_mask_vs_reference_trace_and_oracle(g):
    import oracle
    n = sum(1 for k in g.files if k.startswith("fadd") and k.endswith("_valid"))
    for i in range(n):
        pts = g[f"gftt{int(g[f'fadd{i}_gftt'])}_out"].reshape(-1, 2)
        valid = hotpath.min_distance_mask(pts, g[f"fadd{i}_existing"], float(g[f"fadd{i}_min_dist"]))
        assert valid.dtype == bool and np.array_equal(valid, g[f"fadd{i}_valid"].astype(bool)), i
    rng = np.random.default_rng(5)
    for n, m in ((1400, 3000), (300, 700), (1, 1), (50, 0), (0, 40), (33, 31)):
        pts = np.rint(rng.uniform(0, 1200, (n, 2))).astype(np.float32)
        ex = rng.uniform(0, 1200, (m, 2)).astype(np.float32)
        if n > 1 and m > 1:   # exact ties: distance == 10 is NOT > 10; one float32 step above is
            ex[0] = pts[0] + np.float32([6, 8])
            ex[1] = pts[1] + np.float32([6, np.nextafter(np.float32(8), np.float32(9))])
        ref = np.array([np.all(np.linalg.norm(pts[i, :] - ex, axis=1) > 10) for i in range(n)], bool)        # ref :258
        got = hotpath.min_distance_mask(pts, ex, 10.0)
        assert np.array_equal(got, ref) and np.array_equal(got, oracle.min_distance_mask(pts, ex, 10.0)), (n, m)


def test_triangulate_vs_reference_trace_and_oracle(g):
    import oracle
    n = sum(1 for k in g.files if k.startswith("tri") and k.endswith("_keep"))
    assert n >= 4
    for i in range(n):
        args = (g[f"tri{i}_first_keys"], g[f"tri{i}_keys"], g[f"tri{i}_first_pose"], g[f"tri{i}_poses"])
        keep, lm, kp = hotpath.triangulate_landmarks(g["K"], OPT(g["tri_cfg"]), *args, g[f"tri{i}_cur"][:9].reshape(3, 3), g[f"tri{i}_cur"][9:])
        assert np.array_equal(keep, g[f"tri{i}_keep"].astype(bool)), f"tri{i}: too_short_baseline"
        ref = g[f"tri{i}_landmarks"].reshape(-1, 3)
        assert lm.shape == ref.shape and lm.dtype == np.float32
        assert np.array_equal(kp, g[f"tri{i}_keypoints"].reshape(-1, 2))
        if len(ref):
            assert np.all(np.abs(lm - ref) <= np.spacing(np.abs(ref))), f"tri{i}: landmarks vs the reference's"      # <= 1 float32 ulp
        ko, lo, po = oracle.triangulate_landmarks(g["K"], g["tri_cfg"], *args, g[f"tri{i}_cur"])
        assert np.array_equal(keep, ko) and np.array_equal(kp, po)
        assert np.array_equal(lm, lo), f"tri{i}: landmarks vs the oracle (same arithmetic: bit-equal)"


def test_triangulate_edges():
    K = np.array([[718.856, 0, 607.1928], [0, 718.856, 185.2157], [0, 0, 1]])
    opt = dict(min_dist_landmarks=1, max_dist_landmarks=150, min_baseline_angle=2, min_baseline_frames=2)
    keep, lm, kp = hotpath.triangulate_landmarks(K, opt, np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32), np.zeros((0, 1)),
                                                 [(np.eye(3), np.zeros((3, 1)))], np.eye(3), np.zeros((3, 1)))
    assert keep.shape == (0,) and lm.shape == (0, 3) and kp.shape == (0, 2)
    # identical poses: zero parallax -> every candidate stays (too short baseline), nothing is appended
    pts = np.float32([[100, 100], [640, 180], [900, 300]])
    keep, lm, kp = hotpath.triangulate_landmarks(K, opt, pts, pts, np.zeros(3), [(np.eye(3), np.zeros((3, 1)))], np.eye(3), np.zeros((3, 1)))
    assert keep.all() and len(lm) == 0
    with pytest.raises(Exception):
        hotpath.triangulate_landmarks(K, dict(opt, min_baseline_frames=-5), pts, pts, np.full(3, 7), [(np.eye(3), np.zeros((3, 1)))],
                                      np.eye(3), np.zeros((3, 1)))


def test_recover_pose_vs_oracle_and_live_cv2(g):
    """ref :315 through the cv2-shaped shim: count, 0/255 mask and (R, t) vs the oracle, the recorded call and live cv2."""
    import sys
    import oracle
    sys.path.insert(0, GOLDEN)
    from make_golden import make_emat_pair
    good, R, t, mask = cv2_compat.recoverPose(g["rpose0_E"], g["rpose0_p1"], g["rpose0_p2"], g["K"])
    assert good == int(g["rpose0_good"]) and np.array_equal(mask, g["rpose0_mask"]) and mask.shape == g["rpose0_mask"].shape
    assert R.shape == (3, 3) and t.shape == (3, 1) and np.abs(R - g["rpose0_R"]).max() < 1e-12 and np.abs(t - g["rpose0_t"]).max() < 1e-12
    for n, of, seed in ((600, 0.2, 7), (2500, 0.3, 40), (300, 0.6, 3), (50, 0.0, 9), (5, 0.0, 2)):
        p1, p2, K = make_emat_pair(n, of, seed)
        E, _ = cv2_compat.findEssentialMat(p1, p2, K, method=cv2_compat.RANSAC, prob=0.99, threshold=1)
        good, R, t, mask = cv2_compat.recoverPose(E, p1, p2, K)
        go, Ro, to, mo = oracle.recover_pose(E, p1, p2, K)
        assert good == go and np.array_equal(mask, mo)
        assert np.abs(R - Ro).max() < 1e-14 and np.abs(t - to).max() < 1e-14     # same algorithm; libm hypot/sqrt may differ in the last bit
        try:
            import cv2
        except ImportError:
            continue
        gc, Rc, tc, mc = cv2.recoverPose(E, p1, p2, K)
        assert good == gc and np.array_equal(mask, mc) and np.abs(R - Rc).max() < 1e-12 and np.abs(t - tc).max() < 1e-12
    with pytest.raises(NotImplementedError):
        cv2_compat.recoverPose(E, p1, p2)


def test_batched_forms_vs_oracle(g):
    """SURVEY 8f, "batched f1/f2": one or two launches for a whole batch of sequences, ragged counts; every sequence
    gives what the oracle gives for it alone (the per-sequence entry points are the batch of one)."""
    import oracle
    rng = np.random.default_rng(11)
    # ---- f2: ragged sets, planted exact ties ----
    batch, n_cap, m_cap = 7, 96, 160
    n = np.array([96, 0, 40, 1, 77, 96, 13], np.int32)
    m = np.array([160, 50, 0, 1, 160, 31, 99], np.int32)
    pts = np.rint(rng.uniform(0, 600, (batch, n_cap, 2))).astype(np.float32)
    ex = rng.uniform(0, 600, (batch, m_cap, 2)).astype(np.float32)
    ex[0, 0] = pts[0, 0] + np.float32([6, 8])                                                   # distance == 10: not > 10
    ex[4, 1] = pts[4, 1] + np.float32([6, np.nextafter(np.float32(8), np.float32(9))])           # one step above
    got = hotpath.batch_min_distance_mask(pts, n, ex, m, 10.0)
    assert got.shape == (batch, n_cap) and got.dtype == bool
    for s in range(batch):
        want = oracle.min_distance_mask(pts[s, :n[s]], ex[s, :m[s]], 10.0)
        assert np.array_equal(got[s, :n[s]], want) and not got[s, n[s]:].any(), s
    # ---- f1: the recorded reference calls as sequences of one batch (different candidate counts and pose histories) ----
    nt = sum(1 for k in g.files if k.startswith("tri") and k.endswith("_keep"))
    seqs = list(range(nt)) + [0]                                   # one sequence twice, truncated the second time
    cap = max(len(g[f"tri{i}_keys"]) for i in range(nt)) + 5
    pose_cap = max(len(g[f"tri{i}_poses"]) for i in range(nt)) + 2
    B = len(seqs)
    fk = np.zeros((B, cap, 2), np.float32); k = np.zeros((B, cap, 2), np.float32); fp = np.zeros((B, cap), np.int32)
    nn = np.zeros(B, np.int32); poses = np.zeros((B, pose_cap, 12)); npz = np.zeros(B, np.int32); cur = np.zeros((B, 12))
    for s, i in enumerate(seqs):
        cnt = len(g[f"tri{i}_keys"]) if s < nt else 37
        fk[s, :cnt] = g[f"tri{i}_first_keys"].reshape(-1, 2)[:cnt]; k[s, :cnt] = g[f"tri{i}_keys"].reshape(-1, 2)[:cnt]
        fp[s, :cnt] = np.asarray(g[f"tri{i}_first_pose"]).reshape(-1)[:cnt]
        nn[s] = cnt
        P = np.asarray(g[f"tri{i}_poses"]).reshape(-1, 12)
        poses[s, :len(P)] = P; npz[s] = len(P); cur[s] = g[f"tri{i}_cur"]
    keep, lm, kp, n_new = hotpath.batch_triangulate_landmarks(g["K"], OPT(g["tri_cfg"]), fk, k, fp, nn, poses, npz, cur)
    for s, i in enumerate(seqs):
        cnt = int(nn[s])
        wk, wl, wp = oracle.triangulate_landmarks(g["K"], g["tri_cfg"], fk[s, :cnt], k[s, :cnt], fp[s, :cnt], poses[s, :npz[s]], cur[s])
        assert np.array_equal(keep[s, :cnt], wk) and int(n_new[s]) == len(wl), s
        assert np.array_equal(lm[s, :n_new[s]], wl) and np.array_equal(kp[s, :n_new[s]], wp), s
