"""Lens distortion on the device: cv2_compat.undistort against cv2 and the oracle (tests/undistort_reference.py), and the
per-sequence distortion of SequenceBatch / VOBatch (set_distortion): a sequence with distortion computes bit for bit what a
batch without distortion computes on its cv2.undistort-ed frames, and every other sequence what it computes in a batch
without any distortion."""
import numpy as np
import pytest

import undistort_reference as U
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT
from monocular_visual_odometry_va4mr_b200 import cv2_compat, synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch, initial_state, match_bootstrap_frames

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
MILD = [[-0.06, 0.01, 0.0004, -0.0003, 0.0], [0.04, -0.01, 0.0, 0.0], [-0.05, 0.02, 0.0002, 0.0001, 0.0, 0.01, 0.004, 0.001]]


# ---------------------------------------------------------------- per call
@pytest.mark.parametrize("cam", list(U.CAMERAS))
@pytest.mark.parametrize("model", list(U.MODELS))
def test_undistort_per_call(cam, model):
    K, rows, cols = U.CAMERAS[cam]
    img = synth.render_sequence(cam, 1, seed=len(model))["frames"][0]
    assert img.shape == (rows, cols)
    got = cv2_compat.undistort(img, K, np.asarray(U.MODELS[model]))
    assert np.array_equal(got, cv2.undistort(img, K, np.asarray(U.MODELS[model], np.float64)))
    assert np.array_equal(got, U.undistort(img, K, U.MODELS[model]))


@pytest.mark.parametrize("rows,cols,frac", [(16, 16, (0.0, 0.0)), (17, 23, (0.5, 0.25)), (97, 131, (0.3125, -0.71875)),
                                            (480, 640, (0.1, 0.9))])
def test_undistort_per_call_small_and_fractional(rows, cols, frac):
    K0, r0, c0 = U.CAMERAS["parking"]
    K = U.scale_K(K0, rows, cols, r0, c0, frac)
    rng = np.random.default_rng(rows)
    img = rng.integers(0, 256, (rows, cols), dtype=np.uint8)
    for model in ("plumb_4", "pincushion_5", "rational_pole_8"):
        d = np.asarray(U.MODELS[model])
        got = cv2_compat.undistort(img, K, d)
        assert np.array_equal(got, cv2.undistort(img, K, d)) and np.array_equal(got, U.undistort(img, K, d)), model
    strided = np.zeros((rows, cols + 7), np.uint8)
    strided[:, :cols] = img
    assert np.array_equal(cv2_compat.undistort(strided[:, :cols], K, d), U.undistort(img, K, d))


def test_undistort_refusals():
    K, rows, cols = U.CAMERAS["parking"]
    img = np.zeros((rows, cols), np.uint8)
    d = np.asarray(U.MODELS["plumb_4"])
    for kwargs in (dict(newCameraMatrix=K * 2), ):
        with pytest.raises(NotImplementedError):
            cv2_compat.undistort(img, K, d, **kwargs)
    assert np.array_equal(cv2_compat.undistort(img, K, d, newCameraMatrix=K), U.undistort(img, K, d))
    with pytest.raises(NotImplementedError):
        cv2_compat.undistort(np.zeros((rows, cols, 3), np.uint8), K, d)
    for n in (12, 14):
        with pytest.raises(NotImplementedError):
            cv2_compat.undistort(img, K, np.zeros(n))
    skew = K.copy()
    skew[0, 1] = 0.5
    with pytest.raises(NotImplementedError):
        cv2_compat.undistort(img, skew, d)
    for bad in (np.array([np.nan, 0, 0, 0]), np.array([0, np.inf, 0, 0, 0]), np.zeros(6), np.zeros(3)):
        with pytest.raises(cv2_compat.error):
            cv2_compat.undistort(img, K, bad)
    with pytest.raises(cv2_compat.error):
        cv2_compat.undistort(img, np.diag([0.0, 1.0, 1.0]), d)
    with pytest.raises(cv2_compat.error):
        cv2_compat.undistort(img.astype(np.float32), K, d)


# ---------------------------------------------------------------- SequenceBatch
KITTI = [(synth.K_KITTI, (376, 1241)), (np.array([[721.5377, 0, 609.5593], [0, 721.5377, 172.854], [0, 0, 1.0]]), (375, 1242)),
         (np.array([[707.0912, 0, 601.8873], [0, 707.0912, 183.1104], [0, 0, 1.0]]), (370, 1226))]
SLOT = (376, 1242)


def test_sequence_batch_distortion_equals_undistorted_input():
    """Distorted and undistorted sequences at mixed sizes and cameras against a batch without distortion fed the
    cv2.undistort-ed frames: host steps, submitted frames, good_features, and a prime after set_distortion(None)."""
    n, n_steps = 6, 5
    seqs = []
    for i in range(n):
        K, (r, c) = KITTI[i % 3]
        s = synth.render_sequence("kitti", n_steps + 1, seed=40 + i, width=c, height=r, K=K)
        d = MILD[i % 3] if i % 2 == 0 else None
        seqs.append((s, K, (r, c), d))
    Ks = np.stack([K for _, K, _, _ in seqs])
    sizes = [sz for _, _, sz, _ in seqs]
    dist = [d for *_, d in seqs]
    und = [[U.undistort(f, K, d) if d is not None else f for f in s["frames"]] for s, K, _, d in seqs]
    raw = [list(s["frames"]) for s, *_ in seqs]
    L = 400
    pts = np.zeros((n, L, 2), np.float32)
    obj = np.zeros((n, L, 3), np.float32)
    n_lm = np.zeros(n, np.int32)
    for k, (s, K, _, _) in enumerate(seqs):
        p = synth.grid_corners(und[k][0], L, seed=k).astype(np.float32)[:L]
        o = synth.backproject(K, s["R_cw"][0], s["c"][0], p.astype(np.float64), s["depth"][0]).astype(np.float32)
        pts[k, :len(p)], obj[k, :len(p)], n_lm[k] = p, o, len(p)
    d_rows = np.array([U.dist8(d) for d in dist])
    a = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, dist_coeffs=[U.dist8(d)[:8] for d in dist], max_landmarks=L, max_candidates=L)
    b = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, max_landmarks=L, max_candidates=L)
    assert np.array_equal(a.dist_coeffs, d_rows) and not b.dist_coeffs.any()

    def same_outputs(ra, rb):
        for key in ("lm_next", "lm_status", "cand_next", "cand_status", "pose", "pnp_ok", "inlier_mask", "n_inliers"):
            assert np.array_equal(ra[key], rb[key], equal_nan=True), key

    def same_features():
        ca, na = a.good_features(1400, 0.1, 10.0)
        cb, nb = b.good_features(1400, 0.1, 10.0)
        assert np.array_equal(na, nb) and np.array_equal(ca, cb)

    a.prime([f[0] for f in raw])
    b.prime([f[0] for f in und])
    same_features()
    for t in range(1, n_steps + 1):
        if t % 2:
            ra = {k: v.copy() for k, v in a.step([f[t] for f in raw], pts, obj, n_lm, pts, n_lm).items()}
            rb = b.step([f[t] for f in und], pts, obj, n_lm, pts, n_lm)
        else:
            a.submit_frames([f[t] for f in raw])
            b.submit_frames([f[t] for f in und])
            ra = {k: v.copy() for k, v in a.step(None, pts, obj, n_lm, pts, n_lm).items()}
            rb = b.step(None, pts, obj, n_lm, pts, n_lm)
        same_outputs(ra, rb)
        same_features()
    # cleared: the raw frames again
    a.set_distortion(np.arange(n), None)
    assert not a.dist_coeffs.any()
    a.prime([f[0] for f in raw])
    b.prime([f[0] for f in raw])
    same_features()
    ra = {k: v.copy() for k, v in a.step([f[1] for f in raw], pts, obj, n_lm, pts, n_lm).items()}
    same_outputs(ra, b.step([f[1] for f in raw], pts, obj, n_lm, pts, n_lm))
    a.close()
    b.close()


# ---------------------------------------------------------------- VOBatch
CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
CAMS = ["kitti", "malaga", "parking"]
VSLOT = (768, 1241)
N_FRAMES = 26
DISTORTED = [0, 2, 4]
MASKED = [0, 1]
# after the bootstrap on frames 0 and 2: full steps, listed steps, step_dev with submitted sets, then set_distortion(None)
# ("clear": the sequences become IDLE and are loaded again with their states) and full steps on raw frames
SCHEDULE = ([("full", None)] * 5 + [("listed", [4, 1, 0]), ("listed", [2, 3, 5]), ("listed", [5, 0]), ("listed", [1, 2, 3, 4])]
            + [("dev", None)] * 5 + [("listed", [0, 1, 2, 3, 4, 5])] + [("clear", None)] + [("full", None)] * 4)


@pytest.fixture(scope="module")
def scenes():
    out = []
    for i in range(6):
        cam = CAMS[i // 2]
        K, rows, cols = U.CAMERAS[cam]
        s = synth.render_sequence(cam, N_FRAMES, seed=700 + i)
        d = MILD[i // 2] if i in DISTORTED else None
        mask = None
        if i in MASKED:
            mask = np.full((rows, cols), 255, np.uint8)
            mask[-rows // 6:] = 0   # a hood
        out.append(dict(raw=s["frames"], K=K, size=(rows, cols), dist=d, mask=mask,
                        und=[U.undistort(f, K, d) for f in s["frames"]] if d is not None else s["frames"]))
    return out


def _slot(images):
    out = np.zeros((len(images),) + VSLOT, np.uint8)
    for k, im in enumerate(images):
        out[k, :im.shape[0], :im.shape[1]] = im
    return out


def _refusals(vb, scenes):
    """every bad set_distortion raises and changes nothing"""
    before, status = vb.dist_coeffs.copy(), [vb.read_state(s)["status"] for s in range(len(scenes))]
    good = np.array(MILD[0][:4])
    for seqs, dist in (([0, 0], [good, good]), ([6], [good]), ([-1], [good]), ([], np.zeros((0, 4))), ([[0]], [good]),
                       ([0, 2], [good]), ([0], np.zeros((1, 6))), ([0], np.zeros((1, 3))), ([0], np.zeros(4)),
                       ([0, 1], [good, [np.nan, 0, 0, 0]]), ([1], [[0, np.inf, 0, 0, 0]])):
        with pytest.raises(ValueError):
            vb.set_distortion(seqs, dist)
    with pytest.raises(NotImplementedError):
        vb.set_distortion([0], np.zeros((1, 12)))
    assert np.array_equal(vb.dist_coeffs, before)
    assert [vb.read_state(s)["status"] for s in range(len(scenes))] == status


def _run(scenes, distorted):
    """One VOBatch of the scenes following SCHEDULE.  distorted: the sequences with distortion get raw frames and
    set_distortion; otherwise every sequence gets the undistorted frames (the raw ones after "clear").
    -> (bootstrap result, per sequence the (result row, state) of every advance)"""
    import torch
    n = len(scenes)
    vb = VOBatch(n, *VSLOT, np.stack([sc["K"] for sc in scenes]), OPT, frame_size=[sc["size"] for sc in scenes], **CAPS)
    vb.set_detection_mask(MASKED, [scenes[s]["mask"] for s in MASKED])
    key = "raw" if distorted else "und"
    if distorted:
        _refusals(vb, scenes)
        vb.set_distortion(DISTORTED, [U.dist8(scenes[s]["dist"]) for s in DISTORTED])
        assert list(np.flatnonzero(vb.dist_coeffs.any(1))) == DISTORTED
        assert all(vb.read_state(s)["status"] == VOBatch.IDLE for s in DISTORTED)
        _refusals(vb, scenes)
    boot = {k: np.array(v) for k, v in vb.bootstrap([sc[key][0] for sc in scenes], [sc[key][2] for sc in scenes]).items()}
    nxt = [3] * n
    log = [[(None, vb.read_state(s))] for s in range(n)]
    dev_frames = []
    z = lambda *shape, dt=torch.int32: torch.zeros(shape, dtype=dt, device="cuda")
    out = dict(status=z(n), n_inliers=z(n), n_lm=z(n), n_cand=z(n), pose_cw=z(n, 12, dt=torch.float64))
    for form, seqs in SCHEDULE:
        if form == "clear":
            states = [vb.read_state(s) for s in DISTORTED]
            if distorted:
                vb.set_distortion(DISTORTED, None)
                assert not vb.dist_coeffs.any()
                assert all(vb.read_state(s)["status"] == VOBatch.IDLE for s in DISTORTED)
            key = "raw"
            for s, st in zip(DISTORTED, states):
                vb.load(s, scenes[s][key][nxt[s] - 1], st)
            continue
        listed = list(range(n)) if seqs is None else seqs
        images = [scenes[s][key][nxt[s]] for s in listed]
        if form == "full":
            r = {k: np.array(v) for k, v in vb.step(images).items()}
        elif form == "listed":
            r = {k: np.array(v) for k, v in vb.step(images, seqs=seqs).items()}
        else:
            f = torch.from_numpy(_slot(images)).cuda()
            torch.cuda.synchronize()
            dev_frames.append(f)
            vb.submit_frames_dev(f.data_ptr())
            if distorted and len(dev_frames) == 1:   # refused while a submitted set waits, and nothing changes
                with pytest.raises(ValueError):
                    vb.set_distortion([DISTORTED[0]], None)
                with pytest.raises(ValueError):
                    vb.set_intrinsics([DISTORTED[0]], scenes[DISTORTED[0]]["K"][None])
                vb.set_intrinsics([1], scenes[1]["K"][None])   # a sequence without distortion keeps today's behaviour
                assert vb.dist_coeffs[DISTORTED[0]].any()
            vb.step_dev(None, {k: v.data_ptr() for k, v in out.items()})
            vb.ctx.sync()
            r = {k: v.cpu().numpy() for k, v in out.items()}
        for row, s in enumerate(listed):
            log[s].append(({k: r[k][row].copy() for k in r}, vb.read_state(s)))
            nxt[s] += 1
    vb.close()
    return boot, log


def test_vobatch_distortion(scenes):
    boot, log = _run(scenes, True)
    ref_boot, ref_log = _run(scenes, False)
    for s in range(len(scenes)):
        for k in boot:
            assert boot[k][s] == ref_boot[k][s], (s, k)
        assert boot["status"][s] == VOBatch.OK, s
        assert len(log[s]) == len(ref_log[s])
        for (ra, sa), (rb, sb) in zip(log[s], ref_log[s]):
            if ra is not None:
                for k in ra:
                    assert np.array_equal(ra[k], rb[k], equal_nan=True), (s, k)
            for k in STATE_KEYS:
                assert np.array_equal(sa[k], sb[k], equal_nan=True), (s, k)
            assert sa["status"] == sb["status"], s
    live = sum(log[s][-1][1]["status"] == VOBatch.OK for s in range(len(scenes)))
    assert live >= 4, "too few sequences stayed live for the comparison to mean much"


def test_vobatch_load_with_K_on_a_distorted_sequence(scenes):
    """load(K=) puts K in place before the frame is undistorted: the same pyramid as set_intrinsics then load"""
    sc = scenes[0]
    K2 = sc["K"].copy()
    K2[0, 2] += 3.0
    st = initial_state(sc["K"], OPT, *match_bootstrap_frames(sc["und"][0], sc["und"][2], OPT["feature_ratio"]))
    st = {k: st[k] for k in STATE_KEYS}
    res = []
    for via_K in (True, False):
        vb = VOBatch(1, *VSLOT, sc["K"], OPT, frame_size=[sc["size"]], dist_coeffs=[U.dist8(sc["dist"])], **CAPS)
        with pytest.raises(ValueError):   # a refused load leaves K as it was
            vb.load(0, sc["raw"][2], dict(st, first_pose=np.full(len(st["keys"]), 5, np.int32)), K=K2)
        assert np.array_equal(vb.read_state(0)["status"], VOBatch.IDLE)
        if via_K:
            vb.load(0, sc["raw"][2], st, K=K2)
        else:
            vb.set_intrinsics([0], K2[None])
            vb.load(0, sc["raw"][2], st)
        r = {k: np.array(v) for k, v in vb.step([sc["raw"][3]]).items()}
        res.append([r[k] for k in sorted(r)] + [vb.read_state(0)[k] for k in STATE_KEYS])
        vb.close()
    assert all(np.array_equal(x, y, equal_nan=True) for x, y in zip(*res))
    assert res[0][sorted(r).index("status")][0] == VOBatch.OK
