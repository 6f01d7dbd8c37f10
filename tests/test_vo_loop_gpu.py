"""The device-resident per-frame loop (batch.VOBatch, b200vo_loop_*): one step per frame for a batch of sequences must
follow the data flow of tests/mini_vo.py `MiniVO.step` exactly, as the per-call CUDA entry points compute it."""
import numpy as np
import pytest

from mini_vo import REFERENCE_KITTI_OPTIONS as OPT, rodrigues
from monocular_visual_odometry_va4mr_b200 import cv2_compat, hotpath, synth
from monocular_visual_odometry_va4mr_b200.batch import VOBatch, initial_state, match_bootstrap_frames

pytestmark = pytest.mark.gpu

CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")


@pytest.fixture(scope="module")
def scenes():
    """Six KITTI-shaped sequences from different render seeds, each bootstrapped on frames 0 and 2."""
    out = []
    for seed in range(6):
        s = synth.render_sequence("kitti", 15, seed=100 + seed)
        st = initial_state(s["K"], OPT, *match_bootstrap_frames(s["frames"][0], s["frames"][2], OPT["feature_ratio"]))
        out.append((s["frames"], st))
    return s["K"], out


def _percall_step(st, prev, img, K, pose_cw):
    """MiniVO.step on the per-call entry points.  Returns (status, n_inliers, host pose (12,), new state); the new pose
    of the state is `pose_cw` (the loop's), so that an ulp of sin / cos does not accumulate."""
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


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def test_loop_equals_per_call_path(scenes):
    K, seqs = scenes
    vb = VOBatch(len(seqs), 376, 1241, K, OPT, **CAPS)
    for s, (frames, st) in enumerate(seqs):
        vb.load(s, frames[2], st)
    ref = [dict((k, st[k]) for k in STATE_KEYS) for _, st in seqs]
    live = [True] * len(seqs)
    for f in range(3, 15):
        r = vb.step(np.stack([fr[f] for fr, _ in seqs]))
        for s, (frames, _) in enumerate(seqs):
            if not live[s]:
                assert r["status"][s] != VOBatch.OK
                continue
            code, n_inl, host, new = _percall_step(ref[s], frames[f - 1], frames[f], K, r["pose_cw"][s].copy())
            assert r["status"][s] == code, (s, f)
            assert r["n_inliers"][s] == n_inl, (s, f)
            if code != VOBatch.OK:
                live[s] = False
                continue
            assert np.abs(r["pose_cw"][s] - host).max() <= 1e-12, (s, f)
            assert r["n_lm"][s] == len(new["lm"]) and r["n_cand"][s] == len(new["keys"]), (s, f)
            _assert_state(vb.read_state(s), new)
            ref[s] = new
    assert sum(live) >= 4, "too few sequences ran all 12 steps for the comparison to mean much"


def test_reference_run():
    """Bootstrapped from the recorded ratio-test survivors, the loop stays as close to the recorded reference run as the
    call-by-call CUDA path does (test_free_running_26_frames_on_cuda_path)."""
    import os
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "reference_long.npz"))
    frames = synth.render_sequence(str(g["render_shape"]), int(g["render_n"]), seed=int(g["render_seed"]))["frames"]
    b1 = int(g["bootstrap"][1])
    st = initial_state(g["K"], OPT, g["p1"], g["p2"])
    vb = VOBatch(1, frames[0].shape[0], frames[0].shape[1], g["K"], OPT, **CAPS)
    vb.load(0, frames[b1], st)
    num_pts = [st["num_pts"]]
    for f in range(b1 + 1, len(frames)):
        r = vb.step(frames[f][None])
        assert r["status"][0] == VOBatch.OK, f
        num_pts.append(int(r["n_inliers"][0]))
    poses = vb.read_state(0)["poses"]
    ref = g["poses"]
    assert poses.shape == ref.shape and len(num_pts) == len(g["num_pts"])
    path = np.concatenate([[0.0], np.cumsum(np.linalg.norm(np.diff(ref[:, 9:], axis=0), axis=1))])
    dev = np.linalg.norm(poses[:, 9:] - ref[:, 9:], axis=1)
    assert np.all(dev[:11] <= 0.005 * np.maximum(path[:11], 1.0)), dev[:11]
    assert np.sqrt((dev ** 2).mean()) <= 0.10 * path[-1], (dev.max(), path[-1])


def _results(r):
    return {k: np.array(v) for k, v in r.items()}


def test_stops_and_isolation(scenes):
    K, seqs = scenes
    (fa, sa), (fb, sb) = seqs[0], seqs[1]
    few = dict(sa, lm=sa["lm"][:7], lm_kp=sa["lm_kp"][:7])
    nan_lm = dict(sa, lm=np.full_like(sa["lm"], np.nan))      # no landmark has a position: every P3P hypothesis is rejected
    C = CAPS["max_candidates"]
    n_dup = C - 4                                              # one candidate, repeated: no room for a frame of corners
    full = dict(sa, keys=np.repeat(sa["keys"][:1], n_dup, 0), first_keys=np.repeat(sa["first_keys"][:1], n_dup, 0),
                first_pose=np.zeros(n_dup, np.int32))
    mixed = VOBatch(6, 376, 1241, K, OPT, **CAPS)              # 0, 1: normal; 2: FEW_POINTS; 3: PNP_FAILED; 4: OVERFLOW; 5: never loaded
    for s, (fr, st) in enumerate([(fa, sa), (fb, sb), (fa, few), (fa, nan_lm), (fa, full)]):
        mixed.load(s, fr[2], st)
    alone = VOBatch(2, 376, 1241, K, OPT, **CAPS)
    alone.load(0, fa[2], sa)
    alone.load(1, fb[2], sb)
    stopped = {}
    for f in range(3, 6):
        frames = np.stack([fa[f], fb[f], fa[f], fa[f], fa[f], fa[f]])
        rm, ra = _results(mixed.step(frames)), _results(alone.step(frames[:2]))
        for k in rm:
            assert np.array_equal(rm[k][:2], ra[k]), k
        assert list(rm["status"][2:]) == [VOBatch.FEW_POINTS, VOBatch.PNP_FAILED, VOBatch.OVERFLOW, VOBatch.IDLE], rm["status"]
        assert not rm["n_inliers"][2:].any() and not rm["pose_cw"][2:].any()
        for s in range(2):
            _assert_state(mixed.read_state(s), alone.read_state(s))
        for s in (2, 3, 4):
            now = mixed.read_state(s)
            if s in stopped:
                _assert_state(now, stopped[s])
            stopped[s] = now
    _assert_state(mixed.read_state(2), few)                   # a stop at the commit leaves the state as it was loaded
    _assert_state(mixed.read_state(3), nan_lm)
    mixed.load(2, fa[5], sa)                                   # load revives a stopped sequence
    r = mixed.step(np.stack([fa[6], fb[6], fa[6], fa[6], fa[6], fa[6]]))
    assert r["status"][2] == VOBatch.OK and r["n_inliers"][2] > 0


def test_forms_agree(scenes):
    import torch
    K, seqs = scenes
    sub = seqs[:2]
    vbs = [VOBatch(2, 376, 1241, K, OPT, **CAPS) for _ in range(3)]
    for vb in vbs:
        for s, (fr, st) in enumerate(sub):
            vb.load(s, fr[2], st)
    host = vbs[1].pinned_frames(5)
    for i, f in enumerate(range(3, 8)):
        host[i] = np.stack([fr[f] for fr, _ in sub])
    dev = torch.from_numpy(np.array(host)).cuda()
    out = dict(status=torch.zeros(2, dtype=torch.int32, device="cuda"), n_inliers=torch.zeros(2, dtype=torch.int32, device="cuda"),
               n_lm=torch.zeros(2, dtype=torch.int32, device="cuda"), n_cand=torch.zeros(2, dtype=torch.int32, device="cuda"),
               pose_cw=torch.zeros((2, 12), dtype=torch.float64, device="cuda"))
    torch.cuda.synchronize()
    vbs[1].submit_frames(host[0])
    vbs[2].submit_frames_dev(dev[0].data_ptr())
    for i in range(5):
        ra = _results(vbs[0].step(np.array(host[i])))
        if i + 1 < 5:
            vbs[1].submit_frames(host[i + 1])
        rb = _results(vbs[1].step(None))
        if i + 1 < 5:
            vbs[2].submit_frames_dev(dev[i + 1].data_ptr())
        vbs[2].step_dev(None, {k: v.data_ptr() for k, v in out.items()})
        vbs[2].ctx.sync()
        rc = {k: v.cpu().numpy() for k, v in out.items()}
        for k in ra:
            assert np.array_equal(ra[k], rb[k]) and np.array_equal(ra[k], rc[k]), (i, k)
        assert (ra["status"] == VOBatch.OK).all()
        for s in range(2):
            _assert_state(vbs[1].read_state(s), vbs[0].read_state(s))
            _assert_state(vbs[2].read_state(s), vbs[0].read_state(s))


def test_load_validation(scenes):
    K, seqs = scenes
    fr, st = seqs[0]
    vb = VOBatch(2, 376, 1241, K, OPT, max_landmarks=1024, max_candidates=2048, max_frames=8)
    vb.load(0, fr[2], st)
    before = vb.read_state(0)
    n0 = vb.ctx.launch_count()
    big = lambda a, n: np.repeat(np.asarray(a)[:1], n, 0)
    bad = [dict(st, lm=big(st["lm"], 1025), lm_kp=big(st["lm_kp"], 1025)),
           dict(st, keys=big(st["keys"], 2049), first_keys=big(st["first_keys"], 2049), first_pose=np.zeros(2049, np.int32)),
           dict(st, poses=st["poses"][:0]),
           dict(st, poses=np.repeat(st["poses"][:1], 9, 0)),
           dict(st, first_pose=np.full(len(st["keys"]), 2, np.int32)),
           dict(st, first_pose=np.full(len(st["keys"]), -1, np.int32))]
    for b in bad:
        with pytest.raises(ValueError):
            vb.load(0, fr[3], b)
    with pytest.raises(ValueError):
        vb.load(2, fr[3], st)
    assert vb.ctx.launch_count() == n0
    _assert_state(vb.read_state(0), before)
    assert vb.read_state(0)["status"] == VOBatch.OK and vb.read_state(1)["status"] == VOBatch.IDLE
