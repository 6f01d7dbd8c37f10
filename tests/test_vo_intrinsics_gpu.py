"""Per-sequence camera intrinsics (VOBatch / SequenceBatch `set_intrinsics`, `K` of shape (batch, 3, 3)): a sequence in a
batch of mixed cameras must compute exactly what it computes in a batch of its own camera, and the per-call entry points
with its K."""
import numpy as np
import pytest

from mini_vo import REFERENCE_KITTI_OPTIONS as OPT, rodrigues
from monocular_visual_odometry_va4mr_b200 import cv2_compat, hotpath, synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch, initial_state, match_bootstrap_frames

pytestmark = pytest.mark.gpu

CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
ROWS, COLS = 376, 1241
N_FRAMES = 15


def _K(fx, fy, cx, cy):
    return np.array([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]])


# the three calibrations of the KITTI odometry sequences (00-02, 03, 04-12)
KS = [_K(718.856, 718.856, 607.1928, 185.2157), _K(721.5377, 721.5377, 609.5593, 172.854), _K(707.0912, 707.0912, 601.8873, 183.1104)]


@pytest.fixture(scope="module")
def scenes():
    """Six KITTI-shaped sequences, two per calibration, each rendered through its own camera."""
    out = []
    for i in range(6):
        K = KS[i // 2]
        s = synth.render_sequence("kitti", N_FRAMES, seed=200 + i, K=K)
        out.append((s["frames"], K))
    return out


def _copy(r):
    return {k: np.array(v) for k, v in r.items()}


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def _boot_frames(seqs, idx=None):
    idx = range(len(seqs)) if idx is None else idx
    return np.stack([seqs[i][0][0] for i in idx]), np.stack([seqs[i][0][2] for i in idx])


@pytest.fixture(scope="module")
def mixed_run(scenes):
    """One VOBatch of the six sequences with their own K: device bootstrap on frames 0 and 2, then 12 steps.  Per step the
    result block and every sequence's state."""
    vb = VOBatch(len(scenes), ROWS, COLS, np.stack([K for _, K in scenes]), OPT, **CAPS)
    boot = _copy(vb.bootstrap(*_boot_frames(scenes)))
    states0 = [vb.read_state(s) for s in range(len(scenes))]
    steps = []
    for f in range(3, N_FRAMES):
        r = _copy(vb.step(np.stack([fr[f] for fr, _ in scenes])))
        steps.append((r, [vb.read_state(s) for s in range(len(scenes))]))
    vb.close()
    return boot, states0, steps


def test_mixed_batch_equals_batches_of_one(scenes, mixed_run):
    boot, states0, steps = mixed_run
    assert list(boot["status"]) == [VOBatch.OK] * len(scenes)
    for s, (frames, K) in enumerate(scenes):
        one = VOBatch(1, ROWS, COLS, K, OPT, **CAPS)
        b1 = _copy(one.bootstrap(frames[0][None], frames[2][None]))
        for k in b1:
            assert b1[k][0] == boot[k][s], (s, k)
        _assert_state(one.read_state(0), states0[s])
        for i, f in enumerate(range(3, N_FRAMES)):
            r1 = _copy(one.step(frames[f][None]))
            r, states = steps[i]
            for k in r1:
                assert np.array_equal(r1[k][0], r[k][s]), (s, f, k)
            got = one.read_state(0)
            assert got["status"] == states[s]["status"], (s, f)
            _assert_state(got, states[s])
        one.close()


def _percall_step(st, prev, img, K, pose_cw):
    """MiniVO.step on the per-call entry points with the camera K (test_vo_loop_gpu.py's helper, K passed through).
    Returns (status, n_inliers, host pose (12,), new state); the new pose of the state is `pose_cw` (the loop's)."""
    o = OPT
    p, s_, _ = cv2_compat.calcOpticalFlowPyrLK(prev, img, st["lm_kp"], None, winSize=o["winSize"], maxLevel=o["maxLevel"],
                                               criteria=o["criteria"])
    tr = s_.ravel() == 1
    lm, kp = st["lm"][tr], p.reshape(-1, 2)[tr]
    keys, fk, fp = st["keys"], st["first_keys"], st["first_pose"]
    if len(keys) > 1:
        pk, cs, _ = cv2_compat.calcOpticalFlowPyrLK(prev, img, keys, None, winSize=o["winSize"], maxLevel=o["maxLevel"],
                                                    criteria=o["criteria"])
        ok_c = cs.ravel() == 1
        keys, fk, fp = pk.reshape(-1, 2)[ok_c], fk[ok_c], fp[ok_c]
    if len(kp) < 8:
        return VOBatch.FEW_POINTS, 0, None, st
    ok, rvec, tvec, inl = cv2_compat.solvePnPRansac(lm, kp, K, np.zeros(4), flags=cv2_compat.SOLVEPNP_P3P, confidence=o["PnP_conf"],
                                                    reprojectionError=o["PnP_error"], iterationsCount=o["PnP_iterations"])
    if not ok:
        return VOBatch.PNP_FAILED, 0, None, st
    m = np.isin(np.arange(len(lm)), np.asarray(inl).ravel())
    lm, kp = lm[m], kp[m]
    R_WC = rodrigues(rvec)
    host = np.hstack([R_WC.T.reshape(9), (-R_WC.T @ np.reshape(tvec, (3, 1))).reshape(3)])
    R_CW, t_CW = pose_cw[:9].reshape(3, 3), pose_cw[9:].reshape(3, 1)
    poses = st["poses"]
    if len(keys) > 1:
        too_short, new_lm, new_kp = hotpath.triangulate_landmarks(K, o, fk, keys, fp, poses, R_CW, t_CW)
        lm, kp = np.concatenate([lm, new_lm]), np.concatenate([kp, new_kp])
        keys, fk, fp = keys[too_short], fk[too_short], fp[too_short]
    c = cv2_compat.goodFeaturesToTrack(img, o["feature_max_corners"], o["feature_quality_level"], o["feature_min_dist"],
                                       blockSize=o["feature_block_size"], useHarrisDetector=False, mask=None)
    c = np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)
    c = c[hotpath.min_distance_mask(c, keys, o["feature_min_dist"])]
    new = dict(lm=lm, lm_kp=kp, keys=np.concatenate([keys, c]), first_keys=np.concatenate([fk, c]),
               first_pose=np.concatenate([fp, np.full(len(c), len(poses), np.int32)]), poses=np.vstack([poses, pose_cw]))
    return VOBatch.OK, len(inl), host, new


def test_mixed_batch_follows_per_call_path(scenes, mixed_run):
    boot, states0, steps = mixed_run
    n_live = 0
    for s, (frames, K) in enumerate(scenes):
        st0 = initial_state(K, OPT, *match_bootstrap_frames(frames[0], frames[2], OPT["feature_ratio"]))
        assert boot["num_pts"][s] == st0["num_pts"], s
        _assert_state(states0[s], st0)
        ref, live = dict((k, st0[k]) for k in STATE_KEYS), True
        for i, f in enumerate(range(3, N_FRAMES)):
            r, states = steps[i]
            if not live:
                assert r["status"][s] != VOBatch.OK
                continue
            code, n_inl, host, new = _percall_step(ref, frames[f - 1], frames[f], K, r["pose_cw"][s].copy())
            assert r["status"][s] == code and r["n_inliers"][s] == n_inl, (s, f)
            if code != VOBatch.OK:
                live = False
                continue
            assert np.abs(r["pose_cw"][s] - host).max() <= 1e-12, (s, f)
            _assert_state(states[s], new)
            ref = new
        n_live += live
    assert n_live >= 4, "too few sequences ran all 12 steps for the comparison to mean much"


def test_uniform_K_two_spellings(scenes):
    sub = scenes[:3]
    K = KS[0]
    a = VOBatch(3, ROWS, COLS, K, OPT, **CAPS)
    b = VOBatch(3, ROWS, COLS, np.stack([K] * 3), OPT, **CAPS)
    ra, rb = _copy(a.bootstrap(*_boot_frames(sub))), _copy(b.bootstrap(*_boot_frames(sub)))
    for k in ra:
        assert np.array_equal(ra[k], rb[k]), k
    for f in range(3, 7):
        frames = np.stack([fr[f] for fr, _ in sub])
        ra, rb = _copy(a.step(frames)), _copy(b.step(frames))
        for k in ra:
            assert np.array_equal(ra[k], rb[k]), (f, k)
        for s in range(3):
            _assert_state(a.read_state(s), b.read_state(s))
    assert (ra["status"] == VOBatch.OK).all()


def test_slot_reuse_with_another_camera(scenes):
    """Sequence 1 stops; its slot is bootstrapped with the frames and camera of sequence 4.  The others stay bit-equal to
    an untouched twin, the revived slot equals a fresh batch of one with the new camera."""
    idx = [0, 1, 2]
    Ks = np.stack([scenes[i][1] for i in idx])
    vb = VOBatch(3, ROWS, COLS, Ks, OPT, **CAPS)
    twin = VOBatch(3, ROWS, COLS, Ks, OPT, **CAPS)
    for x in (vb, twin):
        assert (x.bootstrap(*_boot_frames(scenes, idx))["status"] == VOBatch.OK).all()
    st = vb.read_state(1)
    vb.load(1, scenes[1][0][2], dict(st, lm=st["lm"][:7], lm_kp=st["lm_kp"][:7]))   # too few landmarks: stops at the next step
    frames = np.stack([scenes[i][0][3] for i in idx])
    r, rt = _copy(vb.step(frames)), _copy(twin.step(frames))
    assert r["status"][1] == VOBatch.FEW_POINTS
    for k in r:
        assert np.array_equal(r[k][[0, 2]], rt[k][[0, 2]]), k
    new_frames, new_K = scenes[4]
    assert not np.array_equal(new_K, Ks[1])
    rb = vb.bootstrap(new_frames[0][None], new_frames[2][None], seqs=[1], K=new_K[None])
    one = VOBatch(1, ROWS, COLS, new_K, OPT, **CAPS)
    r1 = one.bootstrap(new_frames[0][None], new_frames[2][None])
    for k in rb:
        assert np.array_equal(rb[k], r1[k]), k
    assert rb["status"][0] == VOBatch.OK
    _assert_state(vb.read_state(1), one.read_state(0))
    for f in range(4, 9):
        own = [scenes[i][0][f] for i in idx]
        r = _copy(vb.step(np.stack([own[0], new_frames[f - 1], own[2]])))
        rt = _copy(twin.step(np.stack(own)))
        r1 = _copy(one.step(new_frames[f - 1][None]))
        for k in r:
            assert np.array_equal(r[k][[0, 2]], rt[k][[0, 2]]), (f, k)
            assert np.array_equal(r[k][1], r1[k][0]), (f, k)
        for s in (0, 2):
            _assert_state(vb.read_state(s), twin.read_state(s))
        _assert_state(vb.read_state(1), one.read_state(0))
    assert r["status"][1] == VOBatch.OK


def test_bootstrap_threshold_follows_K(scenes):
    """One frame pair bootstrapped under two cameras whose (fx + fy) / 2 differ: the essential-matrix threshold in normalised
    coordinates differs, and each slot keeps the inliers findEssentialMat gives for its own K."""
    frames, K0 = scenes[0]
    K1 = _K(540.0, 560.0, 600.0, 180.0)
    vb = VOBatch(2, ROWS, COLS, np.stack([K0, K1]), OPT, **CAPS)
    r = vb.bootstrap(np.stack([frames[0]] * 2), np.stack([frames[2]] * 2))
    p0, p1 = match_bootstrap_frames(frames[0], frames[2], OPT["feature_ratio"])
    for s, K in enumerate((K0, K1)):
        E, mask = cv2_compat.findEssentialMat(p0, p1, K, method=cv2_compat.RANSAC, prob=0.99, threshold=1.0)
        assert E is not None
        inl = mask.ravel() == 1
        assert r["status"][s] == VOBatch.OK and r["num_pts"][s] == int(inl.sum()), s
        # the state is the host chain's with this K, built from these inliers: landmark keypoints + candidates
        got = vb.read_state(s)
        _assert_state(got, initial_state(K, OPT, p0, p1))
        assert len(got["lm_kp"]) + len(got["keys"]) <= int(inl.sum())


def _pose_inputs(n_seq, n_lm, w, h, cap, seed0):
    """Landmarks of frame 0 (rendered depth) and frames 0 / 1 of n_seq small sequences, each rendered through its own camera
    (the three KITTI calibrations scaled to the frame, with a few pixels of offset)."""
    distinct = []
    for j in range(min(n_seq, 6)):
        base = KS[j % 3]
        sc = w / 1241.0
        K = _K(base[0, 0] * sc * (1 + 0.02 * j), base[1, 1] * sc * (1 - 0.01 * j), base[0, 2] * sc + j, base[1, 2] * h / 376.0 - j)
        s = synth.render_sequence("kitti", 2, seed=seed0 + j, width=w, height=h, K=K)
        pts = synth.grid_corners(s["frames"][0], n_lm, seed=j)
        obj = synth.backproject(K, s["R_cw"][0], s["c"][0], pts.astype(np.float64), s["depth"][0]).astype(np.float32)
        distinct.append((K, s["frames"], pts, obj))
    Ks = np.zeros((n_seq, 3, 3))
    f0 = np.zeros((n_seq, h, w), np.uint8)
    f1 = np.zeros_like(f0)
    lm_pts = np.zeros((n_seq, cap, 2), np.float32)
    lm_obj = np.zeros((n_seq, cap, 3), np.float32)
    for i in range(n_seq):
        K, fr, pts, obj = distinct[i % len(distinct)]
        Ks[i], f0[i], f1[i] = K, fr[0], fr[1]
        lm_pts[i, :n_lm], lm_obj[i, :n_lm] = pts, obj
    return Ks, f0, f1, lm_pts, lm_obj


@pytest.mark.parametrize("n_seq,n_lm,cap,w,h", [(5, 300, 320, 480, 200),      # fused pose kernel, one CTA per SM: <1>
                                                 (80, 300, 320, 480, 200),     # fused pose kernel, two CTAs per SM: <2>
                                                 (2, 4200, 4400, 640, 240)])   # more than 4096 landmarks: the separate kernels
def test_sequence_batch_set_intrinsics(n_seq, n_lm, cap, w, h):
    opts = dict(win=(15, 15), max_level=3, criteria=(3, 30, 0.01), pnp_iters=500, pnp_err=8.0, pnp_conf=0.99)
    Ks, f0, f1, lm_pts, lm_obj = _pose_inputs(n_seq, n_lm, w, h, cap, seed0=40)
    sb = SequenceBatch(n_seq, h, w, KS[0], win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                       pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"], max_landmarks=cap,
                       max_candidates=16)
    sb.set_intrinsics(np.arange(n_seq), Ks)
    sb.prime(f0)
    n = np.full(n_seq, n_lm, np.int32)
    o = _copy(sb.step(f1, lm_pts, lm_obj, n, np.zeros((n_seq, 16, 2), np.float32), np.zeros(n_seq, np.int32)))
    fused_one = n_seq == 5   # the same kernel instantiation as the one-call path: the same bits
    for s in range(n_seq):
        keep = o["lm_status"][s, :n_lm] == 1
        ok, rv, tv, inl = cv2_compat.solvePnPRansac(lm_obj[s, :n_lm][keep], o["lm_next"][s, :n_lm][keep], Ks[s], np.zeros(4),
                                                    flags=cv2_compat.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                                                    reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
        assert ok and bool(o["pnp_ok"][s]), s
        mask = np.zeros(cap, np.uint8)
        mask[np.flatnonzero(keep)[inl.ravel()]] = 1
        assert np.array_equal(o["inlier_mask"][s], mask), s
        assert int(o["n_inliers"][s]) == len(inl), s
        pose = np.concatenate([rv.ravel(), tv.ravel()])
        if fused_one:
            assert np.array_equal(o["pose"][s], pose), s
        else:
            assert np.abs(o["pose"][s] - pose).max() <= 1e-9, s
    sb.close()


def test_validation_changes_nothing(scenes):
    idx = [0, 2]
    Ks = np.stack([scenes[i][1] for i in idx])
    vb = VOBatch(2, ROWS, COLS, Ks, OPT, **CAPS)
    twin = VOBatch(2, ROWS, COLS, Ks, OPT, **CAPS)
    for x in (vb, twin):
        assert (x.bootstrap(*_boot_frames(scenes, idx))["status"] == VOBatch.OK).all()
    good = KS[1]

    def with_(i, j, v):
        K = good.copy()
        K[i, j] = v
        return K[None]

    n0 = vb.ctx.launch_count()
    bad = [([0], np.stack([good, good])), ([0], good), ([0, 1], good[None]), ([0], good.reshape(1, 9)),   # shapes
           ([0], with_(0, 0, 0.0)), ([0], with_(0, 0, -700.0)), ([0], with_(1, 1, np.nan)), ([0], with_(0, 0, np.inf)),
           ([0], with_(0, 2, np.nan)), ([1], with_(1, 2, np.inf)),                                        # focal lengths, centre
           ([0], with_(0, 1, 1e-3)), ([0], with_(1, 0, 0.5)),                                              # skew, off-diagonal
           ([0], with_(2, 2, 2.0)), ([1], with_(2, 0, 1e-9)), ([0], with_(2, 1, -1.0)),                   # last row
           ([2], good[None]), ([-1], good[None]), ([0, 0], np.stack([good, good])), ([], np.zeros((0, 3, 3))),   # indices
           ([1, 0], np.stack([good, with_(0, 1, 1.0)[0]]))]                                                # one bad K of two
    for seqs, K in bad:
        with pytest.raises(ValueError):
            vb.set_intrinsics(seqs, K)
    fr = scenes[idx[0]][0]
    with pytest.raises(ValueError):
        vb.load(0, fr[2], vb.read_state(0), K=with_(0, 1, 1.0)[0])
    with pytest.raises(ValueError):
        vb.bootstrap(fr[0][None], fr[2][None], seqs=[0], K=with_(2, 2, 0.0))
    with pytest.raises(ValueError):
        VOBatch(2, ROWS, COLS, np.stack([good] * 3), OPT, **CAPS)
    sb = SequenceBatch(2, 200, 480, good, max_landmarks=64, max_candidates=16)
    with pytest.raises(ValueError):
        sb.set_intrinsics([0, 1], np.stack([good, with_(0, 0, 0.0)[0]]))
    with pytest.raises(ValueError):
        sb.set_intrinsics([3], good[None])
    sb.close()
    assert vb.ctx.launch_count() == n0
    for f in range(3, 6):
        frames = np.stack([scenes[i][0][f] for i in idx])
        r, rt = _copy(vb.step(frames)), _copy(twin.step(frames))
        for k in r:
            assert np.array_equal(r[k], rt[k]), (f, k)
        for s in range(2):
            _assert_state(vb.read_state(s), twin.read_state(s))
    assert (r["status"] == VOBatch.OK).all()


def test_batch_created_before_the_random_table_grows(scenes):
    """A loop created on a fresh context (short table of cv2 random numbers) and then bootstrapped (E-RANSAC's longer draw
    grows the table and moves it) steps exactly as one created afterwards."""
    from monocular_visual_odometry_va4mr_b200 import _lib
    ctx = _lib.Context(0)
    frames, K = scenes[3]
    early = VOBatch(1, ROWS, COLS, K, OPT, ctx=ctx, **CAPS)
    early.bootstrap(frames[0][None], frames[2][None])
    late = VOBatch(1, ROWS, COLS, K, OPT, ctx=ctx, **CAPS)
    late.bootstrap(frames[0][None], frames[2][None])
    for f in range(3, 7):
        re_, rl = _copy(early.step(frames[f][None])), _copy(late.step(frames[f][None]))
        for k in re_:
            assert np.array_equal(re_[k], rl[k]), (f, k)
        _assert_state(early.read_state(0), late.read_state(0))
    assert re_["status"][0] == VOBatch.OK
    early.close()
    late.close()
    ctx.close()
