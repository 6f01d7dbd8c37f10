"""The device loop and the batched detector exactly at, and one past, every capacity limit they have.

The detector ranks at most VO_GFTT_BATCH_CAP = 32768 candidates per image on the batched path; the loop stops a sequence
at that count (DETECT_LIMIT), at `max_landmarks` and `max_candidates` (OVERFLOW on the merge / the corner append), at
`max_frames` (OVERFLOW before anything is written), and runs its pose on the fused kernel up to 4096 correspondences.
Frames with an exact candidate count are a rendered KITTI frame with a dot lattice pasted over most of it (a dot yields two
candidates; a small L-shaped dot of a lower value yields one), tuned on the CPU with `mask_reference.gftt_candidates`.

Every loop case runs the edge sequence in slot 1 of a batch between two normal neighbours, which must compute exactly what
a batch of the two neighbours alone computes.  The edge sequence is checked against an uncapped loop of one sequence (itself
checked against the per-call chain, `_percall_step`) and the capacity rule of INTEGRATION.md §3d: a stop at the commit keeps
the state; an OVERFLOW on the landmark merge keeps the inliers and the filtered candidates; one on the corner append keeps
the landmarks too; neither appends the pose."""
import sys

import numpy as np
import pytest

import mask_reference
import oracle
from conftest import GOLDEN
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT, rodrigues
from monocular_visual_odometry_va4mr_b200 import _lib, cv2_compat, hotpath, synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch, initial_state, match_bootstrap_frames

CAP = 32768                 # VO_GFTT_BATCH_CAP (internal.cuh)
FUSED_MAX_N = 4096          # VO_PNP_FUSED_MAX_N (pnp.cuh)
QUALITY = OPT["feature_quality_level"]
SLOT = (376, 1241)
SMALL = (300, 1100)         # a sequence smaller than the slot: key addresses y * 1100 + x
BIG = dict(max_landmarks=FUSED_MAX_N, max_candidates=16384, max_frames=64)   # the uncapped twin (fused pose kernel too)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")


# ------------------------------------------------------------------------------------------------ lattice frames
def _count(img):
    return len(mask_reference.gftt_candidates(img, QUALITY)[0])


def _paint(base, n_dots, tweak, period=4, dot_rows=None):
    """`base` with rows [8, 8 + 4 * dot_rows + 8) blacked out and `n_dots` 255-dots on a `period` lattice, row-major from the
    top left; `tweak`: a 128-valued L of three pixels under the lattice, which adds one candidate."""
    f = base.copy()
    h, w = f.shape
    ncol = (w - 8) // period
    f[8:8 + period * dot_rows + 8, 4:4 + period * ncol] = 0
    k = np.arange(n_dots)
    f[10 + period * (k // ncol), 6 + period * (k % ncol)] = 255
    if tweak:
        r, c = 8 + period * dot_rows + 3, w // 2
        f[r, c] = f[r, c + 1] = f[r + 1, c] = 128
    return f


def lattice_frame(base, target):
    """`base` with a period-4 dot lattice that gives exactly `target` candidates at QUALITY (deterministic search)."""
    h, w = base.shape
    ncol = (w - 8) // 4
    dot_rows = -(-(target // 2 + 64) // ncol)
    assert 8 + 4 * dot_rows + 8 <= h - 8, "the lattice does not fit the frame"
    guess = target // 2 - 200
    est = guess + (target - _count(_paint(base, guess, False, dot_rows=dot_rows))) // 2
    for n in range(est - 4, est + 5):
        for tweak in (False, True):
            f = _paint(base, n, tweak, dot_rows=dot_rows)
            if _count(f) == target:
                return f
    raise AssertionError(f"no lattice gives {target} candidates")


def plateau_frame(base):
    """A period-3 lattice of 255-dots over 224 x 1237 pixels: equal-valued plateaus, nearly every candidate ties."""
    f = base.copy()
    f[8:232, 2:1239] = 0
    f[10:232:3, 3:1239:3] = 255
    return f


@pytest.fixture(scope="module")
def lattice():
    base = synth.render_sequence("kitti", 4, seed=100)["frames"][3]
    small = synth.render_sequence("kitti", 4, seed=101, width=SMALL[1], height=SMALL[0])["frames"][3]
    out = {n: lattice_frame(base, n) for n in (CAP - 1, CAP, CAP + 1)}
    out["small"] = lattice_frame(small, CAP)
    out["plateau"] = plateau_frame(base)
    out["base"] = base
    return out


def test_lattice_frames_hold_the_counts(lattice):
    """The counts the GPU cases rest on (CPU): exact candidate counts around the cap, the pasted lattice setting the
    maximum eigenvalue (and so the threshold), and a plateau frame far above the cap whose candidates mostly tie."""
    base = lattice["base"]
    assert _count(base) < 2000
    for n in (CAP - 1, CAP, CAP + 1):
        f = lattice[n]
        assert f.shape == SLOT and _count(f) == n
        eig = oracle.min_eig_map(f, 3)
        assert eig.max() > 1.5 * oracle.min_eig_map(base, 3).max()
        r, c = np.unravel_index(np.argmax(eig), eig.shape)
        assert (f != base)[max(r - 2, 0):r + 3, max(c - 2, 0):c + 3].any(), "the maximum is not set by the pasted lattice"
    assert lattice["small"].shape == SMALL and _count(lattice["small"]) == CAP
    idx, w = mask_reference.gftt_candidates(lattice["plateau"], QUALITY)
    vals = oracle.min_eig_map(lattice["plateau"], 3).ravel()[idx]
    assert len(idx) > 8 * CAP and len(np.unique(vals)) * 100 < len(idx)


# ------------------------------------------------------------------------------------------------ detector at the cap
def _want(img, max_corners, min_dist):
    w = mask_reference.good_features_to_track(img, max_corners, QUALITY, min_dist)
    return np.zeros((0, 2), np.float32) if w is None else w.reshape(-1, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("min_dist,max_corners", [(10.0, 1400), (7.0, 20000)])
def test_batched_detector_at_the_cap(lattice, min_dist, max_corners):
    nb = synth.render_sequence("kitti", 4, seed=102)["frames"][3], synth.render_sequence("kitti", 4, seed=103)["frames"][2]
    images = [nb[0], lattice[CAP - 1], lattice["small"], lattice[CAP], nb[1]]
    sizes = [SLOT, SLOT, SMALL, SLOT, SLOT]
    sb = SequenceBatch(5, *SLOT, synth.K_KITTI, max_landmarks=4, max_candidates=0, frame_size=sizes)
    sb.prime(images)
    corners, n = sb.good_features(max_corners, QUALITY, min_dist)
    alone = SequenceBatch(2, *SLOT, synth.K_KITTI, max_landmarks=4, max_candidates=0)
    alone.prime(np.stack(nb))
    ca, na = alone.good_features(max_corners, QUALITY, min_dist)
    assert np.array_equal(n[[0, 4]], na) and np.array_equal(corners[[0, 4]], ca)
    for k, img in enumerate(images):
        want = _want(img, max_corners, min_dist)
        assert n[k] == len(want) and np.array_equal(corners[k, :n[k]], want), (k, n[k], len(want))
    assert n[1:4].min() > 1000

    # one past the cap: the call refuses and writes none of its outputs
    sb.prime([nb[0], lattice[CAP], lattice["small"], lattice[CAP + 1], nb[1]])
    c_out = np.full((5, max_corners, 2), -7.0, np.float32)
    n_out = np.full(5, -7, np.int32)
    rc = sb.ctx.lib.b200vo_batch_good_features(sb.h, max_corners, QUALITY, min_dist, c_out.ctypes.data_as(_lib.c_f32p),
                                               n_out.ctypes.data_as(_lib.c_i32p))
    assert rc != 0 and "exceed" in sb.ctx.last_error()
    assert (c_out == -7.0).all() and (n_out == -7).all()
    with pytest.raises(_lib.B200VOError, match="exceed"):
        sb.good_features(max_corners, QUALITY, min_dist)
    sb.close()
    alone.close()


@pytest.mark.gpu
def test_device_detector_at_the_cap(lattice):
    import torch
    ctx = _lib.default_context(0)
    dev = torch.device("cuda", 0)
    o_c = torch.full((1400, 2), -1.0, dtype=torch.float32, device=dev)
    o_n = torch.zeros((1,), dtype=torch.int32, device=dev)
    for count in (CAP, CAP + 1):
        img = torch.from_numpy(lattice[count]).to(dev)
        o_c.fill_(-1.0)
        torch.cuda.synchronize()
        rc = ctx.lib.b200vo_good_features_to_track_dev(ctx.h, img.data_ptr(), SLOT[0], SLOT[1], SLOT[1], 1400, QUALITY, 10.0, 3,
                                                       o_c.data_ptr(), o_n.data_ptr())
        assert rc == 0, ctx.last_error()
        ctx.sync()
        n, got = int(o_n.item()), o_c.cpu().numpy()
        if count == CAP:
            want = _want(lattice[count], 1400, 10.0)
            assert n == len(want) and np.array_equal(got[:n], want) and (got[n:] == 0).all()
        else:
            assert n == -1 and (got == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("frame", [CAP + 1, "plateau"])
def test_per_call_detector_above_the_cap(lattice, frame):
    """Above 32768 candidates the per-call detector sorts bitonically; the greedy minDistance selection reads that order."""
    img = lattice[frame]
    got = cv2_compat.goodFeaturesToTrack(img, 1400, QUALITY, 10, blockSize=3)
    want = oracle.good_features_to_track(img, 1400, QUALITY, 10)
    assert got is not None and got.shape == want.shape and np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------ pose kernel at 4096
def _pose_close(rv, tv, rv0, tv0, tol=1e-6):
    assert np.abs(np.ravel(rv) - np.ravel(rv0)).max() < tol
    assert np.abs(np.ravel(tv) - np.ravel(tv0)).max() < tol * max(1.0, np.abs(tv0).max())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [FUSED_MAX_N - 1, FUSED_MAX_N, FUSED_MAX_N + 1])
def test_per_call_pnp_at_the_fused_limit(n):
    sys.path.insert(0, GOLDEN)
    from make_golden import make_pnp_case
    obj, img, K = make_pnp_case(n, 0.3, 900 + n)
    ok, rv, tv, inl = cv2_compat.solvePnPRansac(obj, img, K, np.zeros(4), flags=cv2_compat.SOLVEPNP_P3P, confidence=0.99,
                                                reprojectionError=8.0, iterationsCount=500)
    rok, rrv, rtv, rinl, _ = oracle.solve_pnp_ransac_p3p(obj, img, K, 500, 8.0, 0.99)
    assert ok and rok and np.array_equal(inl, rinl)
    _pose_close(rv, tv, rrv, rtv)


# ------------------------------------------------------------------------------------------------ the loop
def _percall_step(st, prev, img, K, pose_cw, mask=None):
    """MiniVO.step on the per-call entry points.  Returns (status, n_inliers, host pose (12,), new state); the new pose
    of the state is `pose_cw` (the loop's), so that an ulp of sin / cos does not accumulate.  `mask`: the detection mask."""
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
    c = cv2_compat.good_features_to_track_masked(img, o["feature_max_corners"], o["feature_quality_level"], o["feature_min_dist"],
                                                 mask, blockSize=o["feature_block_size"])
    c = np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)
    c = c[hotpath.min_distance_mask(c, keys, o["feature_min_dist"])]
    new = dict(lm=lm, lm_kp=kp, keys=np.concatenate([keys, c]), first_keys=np.concatenate([fk, c]),
               first_pose=np.concatenate([fp, np.full(len(c), len(poses), np.int32)]), poses=np.vstack([poses, pose_cw]))
    return VOBatch.OK, len(inl), host, new


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def _results(r):
    return {k: np.array(v) for k, v in r.items()}


def _row(r, i):
    return {k: v[i] for k, v in r.items()}


def _state(st):
    return {k: np.asarray(st[k]) for k in STATE_KEYS}


def _trim(st, n_lm=None, n_cand=None):
    st = _state(st)
    if n_lm is not None:
        st["lm"], st["lm_kp"] = st["lm"][:n_lm], st["lm_kp"][:n_lm]
    if n_cand is not None:
        st["keys"], st["first_keys"], st["first_pose"] = st["keys"][:n_cand], st["first_keys"][:n_cand], st["first_pose"][:n_cand]
    return st


def _pad_poses(st, k):
    """k copies of the first pose in front of the history: every index moves by k, nothing else changes"""
    st = _state(st)
    st["poses"] = np.vstack([np.repeat(st["poses"][:1], k, 0), st["poses"]])
    st["first_pose"] = st["first_pose"] + np.int32(k)
    return st


@pytest.fixture(scope="module")
def scenes():
    """Three KITTI-shaped sequences from different render seeds, each bootstrapped on frames 0 and 2; the first (seed 100)
    is the edge sequence, whose frame 3 is the base of the lattice frames."""
    out = []
    for seed in (100, 101, 102):
        s = synth.render_sequence("kitti", 10, seed=seed)
        st = initial_state(s["K"], OPT, *match_bootstrap_frames(s["frames"][0], s["frames"][2], OPT["feature_ratio"]))
        out.append((s["frames"], _state(st)))
    return s["K"], out


@pytest.fixture(scope="module")
def chain(scenes):
    """The edge sequence's states after frames 2 .. 7 in an uncapped loop"""
    K, seqs = scenes
    frames, st = seqs[0]
    vb = VOBatch(1, *SLOT, K, OPT, **BIG)
    vb.load(0, frames[2], st)
    out = {2: st}
    for f in range(3, 8):
        assert vb.step(frames[f][None])["status"][0] == VOBatch.OK, f
        out[f] = _state(vb.read_state(0))
    vb.close()
    return out


def _reference(K, before, prev, img, mask=None):
    """One step of `before` in an uncapped loop of one sequence, checked against the per-call chain.
    -> (result row, state after the step)"""
    tw = VOBatch(1, *SLOT, K, OPT, **BIG)
    if mask is not None:
        tw.set_detection_mask([0], mask[None])
    tw.load(0, prev, before)
    r = _row(_results(tw.step(img[None])), 0)
    after = _state(tw.read_state(0))
    tw.close()
    code, n_inl, host, new = _percall_step(before, prev, img, K, r["pose_cw"].copy(), mask)
    assert r["status"] == code and r["n_inliers"] == n_inl
    if code == VOBatch.OK:
        assert np.abs(r["pose_cw"] - host).max() <= 1e-12
    _assert_state(after, new)
    return r, after


def _capped(r, after, before, L, C, P):
    """The result row and state the capacity rule of INTEGRATION.md §3d gives for a step whose uncapped outcome is
    (r, after) from `before`"""
    zero = dict(n_inliers=0, pose_cw=np.zeros(12))
    if r["status"] != VOBatch.OK:
        return dict(zero, status=r["status"], n_lm=len(before["lm"]), n_cand=len(before["keys"])), before
    n_poses = len(before["poses"])
    if n_poses >= P:
        return dict(zero, status=VOBatch.OVERFLOW, n_lm=len(before["lm"]), n_cand=len(before["keys"])), before
    m = int(r["n_inliers"])
    kept = int((after["first_pose"] < n_poses).sum())   # the corners of this step come last, with first_pose = n_poses
    cand = _trim(after, n_cand=kept)
    if len(after["lm"]) > L:
        want = dict(_trim(cand, n_lm=m), poses=before["poses"])
    elif len(after["keys"]) > C:
        want = dict(cand, poses=before["poses"])
    else:
        return dict(r), after
    return dict(zero, status=VOBatch.OVERFLOW, n_lm=len(want["lm"]), n_cand=len(want["keys"])), want


class Rig:
    """A batch [neighbour 0, edge, neighbour 1] and a batch of the two neighbours alone, with the same capacities."""

    def __init__(self, scenes, caps, neighbour_state=lambda st: st):
        K, seqs = scenes
        self.K, self.caps = K, caps
        self.nb = [(fr, neighbour_state(st)) for fr, st in seqs[1:3]]
        self.vb = VOBatch(3, *SLOT, K, OPT, **caps)
        self.alone = VOBatch(2, *SLOT, K, OPT, **caps)
        for i, (fr, st) in enumerate(self.nb):
            self.vb.load(2 * i, fr[2], st)
            self.alone.load(i, fr[2], st)
        self.f = 2                         # the neighbours' current frame

    def load(self, prev, st):
        self.vb.load(1, prev, st)

    def step(self, img, listed=False):
        """One step (listed: of the edge and neighbour 0 only); -> the edge's result row and state"""
        self.f += 1
        nf = [fr[self.f] for fr, _ in self.nb]
        if listed:
            r = _results(self.vb.step(np.stack([img, nf[0]]), seqs=[1, 0]))
            ra = _results(self.alone.step(nf[0][None], seqs=[0]))
            for k in r:
                assert np.array_equal(r[k][1:2], ra[k][:1]), k
            edge = _row(r, 0)
        else:
            r = _results(self.vb.step(np.stack([nf[0], img, nf[1]])))
            ra = _results(self.alone.step(np.stack(nf)))
            for k in r:
                assert np.array_equal(r[k][[0, 2]], ra[k]), k
            edge = _row(r, 1)
        for i in range(2):
            _assert_state(self.vb.read_state(2 * i), self.alone.read_state(i))
        return edge, _state(self.vb.read_state(1))

    def expect(self, before, prev, img, mask=None):
        """The edge's step from `before` under this rig's capacities; -> (result row, state) it must produce"""
        r, after = _reference(self.K, before, prev, img, mask)
        c = self.caps
        return _capped(r, after, before, c["max_landmarks"], c["max_candidates"], c["max_frames"])

    def check(self, got, want):
        (r, st), (wr, wst) = got, want
        for k in ("status", "n_inliers", "n_lm", "n_cand"):
            assert r[k] == wr[k], (k, r[k], wr[k])
        assert np.array_equal(r["pose_cw"], wr["pose_cw"])
        _assert_state(st, wst)

    def close(self):
        self.vb.close()
        self.alone.close()


CAPS = dict(max_landmarks=FUSED_MAX_N, max_candidates=8192, max_frames=64)


@pytest.mark.gpu
@pytest.mark.parametrize("listed", [False, True])
def test_detect_limit(scenes, lattice, listed):
    K, seqs = scenes
    frames, st = seqs[0]
    rig = Rig(scenes, CAPS)
    rig.load(frames[2], st)
    want = rig.expect(st, frames[2], lattice[CAP])
    assert want[0]["status"] == VOBatch.OK
    rig.check(rig.step(lattice[CAP], listed), want)

    rig.load(frames[2], st)
    r, now = rig.step(lattice[CAP + 1], listed)
    assert r["status"] == VOBatch.DETECT_LIMIT and r["n_inliers"] == 0 and not r["pose_cw"].any()
    assert r["n_lm"] == len(st["lm"]) and r["n_cand"] == len(st["keys"])
    _assert_state(now, st)
    for f in (4, 5):                                   # a stopped sequence stays as it is
        r, now = rig.step(frames[f], listed)
        assert r["status"] == VOBatch.DETECT_LIMIT and r["n_inliers"] == 0 and not r["pose_cw"].any()
        _assert_state(now, st)
    rig.load(frames[2], st)                            # load revives it
    want = rig.expect(st, frames[2], frames[3])
    assert want[0]["status"] == VOBatch.OK
    rig.check(rig.step(frames[3], listed), want)

    # PnP fails and the frame is over the cap: the PnP stop is the one reported
    nan_lm = dict(st, lm=np.full_like(st["lm"], np.nan))
    rig.load(frames[2], nan_lm)
    r, now = rig.step(lattice[CAP + 1], listed)
    assert r["status"] == VOBatch.PNP_FAILED and r["n_inliers"] == 0
    _assert_state(now, nan_lm)
    rig.close()


def _inlier_rows(before, after, m):
    """the rows of before["lm"] that the step kept as inliers (the first m rows of after["lm"], bit-equal positions)"""
    rows = {tuple(v.view(np.uint32)): i for i, v in enumerate(before["lm"])}
    return np.array([rows[tuple(v.view(np.uint32))] for v in after["lm"][:m]], np.int64)


@pytest.mark.gpu
def test_landmark_limit(scenes, chain):
    K, seqs = scenes
    frames = seqs[0][0]
    full = chain[5]
    r, after = _reference(K, full, frames[5], frames[6])
    keep = _inlier_rows(full, after, int(r["n_inliers"]))
    before = dict(full, lm=full["lm"][keep], lm_kp=full["lm_kp"][keep])   # every loaded landmark is an inlier
    r, after = _reference(K, before, frames[5], frames[6])
    m, nn = int(r["n_inliers"]), len(after["lm"]) - int(r["n_inliers"])
    assert r["status"] == VOBatch.OK and nn >= 1 and len(before["lm"]) <= m + nn - 1 and m + nn <= FUSED_MAX_N, (len(before["lm"]), m, nn)
    for L in (m + nn, m + nn - 1):
        caps = dict(CAPS, max_landmarks=L)
        rig = Rig(scenes, caps, lambda st: _trim(st, n_lm=min(len(st["lm"]), L // 3), n_cand=100))
        rig.load(frames[5], before)
        want = rig.expect(before, frames[5], frames[6])
        got = rig.step(frames[6])
        rig.check(got, want)
        if L == m + nn:
            assert got[0]["status"] == VOBatch.OK and got[0]["n_lm"] == L
            rig.check(rig.step(frames[7]), rig.expect(got[1], frames[6], frames[7]))
        else:
            assert got[0]["status"] == VOBatch.OVERFLOW and got[0]["n_lm"] == m
        rig.close()


@pytest.mark.gpu
def test_candidate_limit(scenes):
    K, seqs = scenes
    frames, before = seqs[0]
    r, after = _reference(K, before, frames[2], frames[3])
    n_poses = len(before["poses"])
    kept = int((after["first_pose"] < n_poses).sum())
    corners = len(after["keys"]) - kept
    assert r["status"] == VOBatch.OK and len(before["keys"]) <= kept + corners - 1, (len(before["keys"]), kept, corners)
    for Cn in (kept + corners, kept + corners - 1):
        rig = Rig(scenes, dict(CAPS, max_candidates=Cn), lambda st: _trim(st, n_cand=0))
        rig.load(frames[2], before)
        got = rig.step(frames[3])
        rig.check(got, rig.expect(before, frames[2], frames[3]))
        if Cn == kept + corners:
            assert got[0]["status"] == VOBatch.OK and got[0]["n_cand"] == Cn
            # the tracker, the triangulation and the distance filter at n = max_candidates
            rig.check(rig.step(frames[4]), rig.expect(got[1], frames[3], frames[4]))
        else:
            assert got[0]["status"] == VOBatch.OVERFLOW and got[0]["n_lm"] == len(after["lm"]) and got[0]["n_cand"] == kept
        rig.close()


@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 64])
def test_pose_history_limit(scenes, chain, P):
    """n_poses = P - 1: one step, then OVERFLOW with the state kept; n_poses = P: OVERFLOW at once.  The padded history only
    moves indices, so the step equals the unpadded reference with its indices moved."""
    K, seqs = scenes
    frames, st = seqs[0]
    if P == 2:
        unpadded, k, prev = dict(st, poses=st["poses"][:1]), 0, 2
        neighbour = lambda s: dict(s, poses=s["poses"][:1])
    else:
        unpadded, k, prev = chain[3], P - 1 - len(chain[3]["poses"]), 3
        neighbour = lambda s: s
    before = _pad_poses(unpadded, k)
    assert len(before["poses"]) == P - 1
    rig = Rig(scenes, dict(CAPS, max_frames=P), neighbour)
    for _ in range(prev - 2):                                   # the neighbours' frames follow the edge's
        rig.step(frames[rig.f + 1])
    rig.load(frames[prev], before)
    wr, wst = rig.expect(unpadded, frames[prev], frames[prev + 1])
    assert wr["status"] == VOBatch.OK
    got = rig.step(frames[prev + 1])
    rig.check(got, (wr, _pad_poses(wst, k)))
    full = got[1]
    assert len(full["poses"]) == P and (full["first_pose"] == P - 1).any()
    r, now = rig.step(frames[prev + 2])
    assert r["status"] == VOBatch.OVERFLOW and r["n_inliers"] == 0 and not r["pose_cw"].any()
    _assert_state(now, full)
    if P > 2:   # loaded full, with candidates whose first pose is the last row of the history
        rig.load(frames[prev + 2], full)
        r, now = rig.step(frames[prev + 3])
        assert r["status"] == VOBatch.OVERFLOW and r["n_lm"] == len(full["lm"]) and r["n_cand"] == len(full["keys"])
        _assert_state(now, full)
    rig.close()


@pytest.mark.gpu
def test_fused_pose_kernel_at_its_limit(scenes):
    """4096 live correspondences in a loop of max_landmarks = 4096: landmarks the tracker keeps, repeated"""
    K, seqs = scenes
    frames, st = seqs[0]
    p, s_, _ = cv2_compat.calcOpticalFlowPyrLK(frames[2], frames[3], st["lm_kp"], None, winSize=OPT["winSize"],
                                               maxLevel=OPT["maxLevel"], criteria=OPT["criteria"])
    ok = np.flatnonzero(s_.ravel() == 1)
    rows = np.resize(ok, FUSED_MAX_N)
    before = dict(st, lm=st["lm"][rows], lm_kp=st["lm_kp"][rows])
    before = _trim(before, n_cand=1)
    rig = Rig(scenes, CAPS)
    rig.load(frames[2], before)
    r, now = rig.step(frames[3])
    code, n_inl, host, new = _percall_step(before, frames[2], frames[3], K, r["pose_cw"].copy())
    assert r["status"] == code == VOBatch.OK and r["n_inliers"] == n_inl
    assert np.abs(r["pose_cw"] - host).max() <= 1e-12
    _assert_state(now, new)
    rig.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_cand", [0, 1, 2])
def test_candidate_count_rules(scenes, n_cand):
    """Candidates are tracked and triangulated only when there are more than one.  The edge sequence detects nothing (an
    all-zero mask), so after a step of two candidates of which the tracker drops one, the next step has a single one."""
    K, seqs = scenes
    frames, st = seqs[0]
    _, cs, _ = cv2_compat.calcOpticalFlowPyrLK(frames[2], frames[3], st["keys"], None, winSize=OPT["winSize"],
                                               maxLevel=OPT["maxLevel"], criteria=OPT["criteria"])
    cs = cs.ravel()
    lost = np.flatnonzero(cs != 1)
    drop = st["keys"][lost[:1]] if len(lost) else np.float32([[-40.0, -40.0]])   # outside the frame: never tracked
    keys = np.concatenate([st["keys"][np.flatnonzero(cs == 1)[:1]], drop])[:n_cand]
    before = dict(st, keys=keys, first_keys=keys.copy(), first_pose=np.zeros(len(keys), np.int32))
    mask = np.zeros(SLOT, np.uint8)
    rig = Rig(scenes, CAPS)
    rig.vb.set_detection_mask([1], mask[None])
    rig.load(frames[2], before)
    cur = before
    for f in (3, 4):
        want = rig.expect(cur, frames[f - 1], frames[f], mask)
        assert want[0]["status"] == VOBatch.OK
        got = rig.step(frames[f])
        rig.check(got, want)
        cur = got[1]
        if n_cand == 1 or f == 4:
            assert len(cur["keys"]) == min(n_cand, 1)
    if n_cand:
        assert np.array_equal(cur["keys"], before["keys"][:1]) == (n_cand == 1)
    rig.close()
