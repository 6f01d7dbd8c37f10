"""Fisheye lenses and undistorted cameras other than the raw one on the device: cv2_compat.fisheye_undistort_image and
cv2_compat.undistort(newCameraMatrix=) against cv2 and the oracle (tests/lens_reference.py), and the per-sequence lenses of
SequenceBatch / VOBatch (set_distortion(model=, raw_K=)): a sequence with a lens computes bit for bit what a batch without
lenses computes on the oracle-undistorted frames with K = the sequence's (new) camera."""
import numpy as np
import pytest

import lens_reference as L
import undistort_reference as U
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT
from monocular_visual_odometry_va4mr_b200 import cv2_compat, synth
from monocular_visual_odometry_va4mr_b200._lib import c_f64p, c_i32p
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch

pytestmark = pytest.mark.gpu
cv2 = pytest.importorskip("cv2")

STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
WRAP_D = np.array([0.5, 0.5, 1.0, 5.0])   # a strong lens: with a tiny Knew on a full-size frame, the map leaves int16 and wraps


def _noise(rows, cols, seed):
    return np.random.default_rng(seed).integers(0, 256, (rows, cols), dtype=np.uint8)


# ---------------------------------------------------------------- per call
def _fisheye_cases():
    for cam, (K, D, rows, cols) in L.FISHEYE.items():
        for knew in ("none", "K", 0.0, 0.5, 1.0):
            yield cam, knew


@pytest.mark.parametrize("cam,knew", list(_fisheye_cases()))
def test_fisheye_undistort_per_call(cam, knew):
    K, D, rows, cols = L.FISHEYE[cam]
    Knew = None if knew == "none" else K if knew == "K" else L.fisheye_knew(cv2, K, D, rows, cols, knew)
    img = _noise(rows, cols, rows + cols)
    got = cv2_compat.fisheye_undistort_image(img, K, np.asarray(D))
    if Knew is not None:
        got = cv2_compat.fisheye_undistort_image(img, K, np.asarray(D), Knew=Knew)
    assert np.array_equal(got, cv2.fisheye.undistortImage(img, K, np.asarray(D, np.float64), Knew=Knew))
    assert np.array_equal(got, L.fisheye_undistort(img, K, D, Knew))


@pytest.mark.parametrize("rows,cols,frac", [(16, 16, (0.0, 0.0)), (17, 23, (0.5, 0.25)), (97, 131, (0.3125, -0.71875)),
                                            (800, 848, (0.0, 0.0))])
def test_fisheye_undistort_small_fractional_zero_and_wrapping(rows, cols, frac):
    """K_T265 scaled to the frame (800 x 848 is the camera itself), zero D, a balance Knew and a tiny Knew with a strong
    lens.  At 800 x 848 the last sends most map entries far outside int16, where cv2 stores them wrapped; some wrapped
    entries land inside the image, so a map that saturated them, as the pinhole map does, would give another image."""
    K0, D, r0, c0 = L.FISHEYE["t265"]
    K = U.scale_K(K0, rows, cols, r0, c0, frac)
    img = _noise(rows, cols, rows)
    tiny = np.array([[0.001, 0.0, cols / 2], [0.0, 0.0012, rows / 2], [0.0, 0.0, 1.0]])
    n_wrapped = 0
    for d, Knew in ((D, K), ([0, 0, 0, 0], K), (D, L.fisheye_knew(cv2, K, D, rows, cols, 0.7)), (WRAP_D, tiny)):
        d = np.asarray(d, np.float64)
        got = cv2_compat.fisheye_undistort_image(img, K, d, Knew=Knew)
        assert np.array_equal(got, cv2.fisheye.undistortImage(img, K, d, Knew=Knew))
        assert np.array_equal(got, L.fisheye_undistort(img, K, d, Knew))
        src = L.fisheye_source_px(K, d, Knew, rows, cols)
        wrapped = (np.abs(src) > 32767).any(-1)
        if wrapped.any():
            xy, fr = L.fisheye_map(K, d, Knew, rows, cols)
            assert np.array_equal(xy, ((src + 32768) % 65536 - 32768).astype(np.int16))
            saturated = np.clip(src, -32768, 32767).astype(np.int16)
            assert (L.remap(img, saturated, fr) != got).sum() > 1000, "the case must tell wrapping from saturating"
            n_wrapped += int(wrapped.sum())
    if (rows, cols) == (800, 848):
        assert n_wrapped > 100000
    strided = np.zeros((rows, cols + 5), np.uint8)
    strided[:, :cols] = img
    assert np.array_equal(cv2_compat.fisheye_undistort_image(strided[:, :cols], K, np.asarray(D), Knew=K), L.fisheye_undistort(img, K, D, K))


@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
@pytest.mark.parametrize("model", ["plumb_4", "kitti_like_5", "rational_8"])
@pytest.mark.parametrize("cam", list(U.CAMERAS))
def test_undistort_new_camera_per_call(cam, model, alpha):
    K, rows, cols = U.CAMERAS[cam]
    d = np.asarray(U.MODELS[model], np.float64)
    Knew = L.pinhole_knew(cv2, K, d, rows, cols, alpha)
    img = _noise(rows, cols, len(model))
    got = cv2_compat.undistort(img, K, d, newCameraMatrix=Knew)
    assert np.array_equal(got, cv2.undistort(img, K, d, newCameraMatrix=Knew))
    assert np.array_equal(got, L.undistort_new(img, K, d, Knew))


def test_one_call_refusals():
    K, D, rows, cols = L.FISHEYE["vga"]
    D = np.asarray(D)
    img = np.zeros((rows, cols), np.uint8)
    skew = K.copy()
    skew[0, 1] = 0.5
    for kwargs in (dict(K=skew), dict(Knew=skew), dict(Knew=K * 2), dict(new_size=(cols + 1, rows))):
        with pytest.raises(NotImplementedError):
            cv2_compat.fisheye_undistort_image(img, **dict(dict(K=K, D=D), **kwargs))
    with pytest.raises(NotImplementedError):
        cv2_compat.fisheye_undistort_image(np.zeros((rows, cols, 3), np.uint8), K, D)
    assert np.array_equal(cv2_compat.fisheye_undistort_image(img + 7, K, D, Knew=K, new_size=(cols, rows)), L.fisheye_undistort(img + 7, K, D, K))
    for bad in (dict(D=np.zeros(5)), dict(D=np.array([np.nan, 0, 0, 0])), dict(D=np.array([0, np.inf, 0, 0])),
                dict(K=np.diag([0.0, 1.0, 1.0])), dict(Knew=np.diag([1.0, -1.0, 1.0])), dict(Knew=np.diag([np.nan, 1.0, 1.0])),
                dict(K=np.eye(2))):
        with pytest.raises(cv2_compat.error):
            cv2_compat.fisheye_undistort_image(img, **dict(dict(K=K, D=D), **bad))
    with pytest.raises(cv2_compat.error):
        cv2_compat.fisheye_undistort_image(img.astype(np.float32), K, D)
    d = np.asarray(U.MODELS["plumb_4"])
    for Knew in (skew, K * 2):
        with pytest.raises(NotImplementedError):
            cv2_compat.undistort(img, K, d, newCameraMatrix=Knew)
    for Knew in (np.diag([0.0, 1.0, 1.0]), np.diag([np.inf, 1.0, 1.0]), np.eye(2)):
        with pytest.raises(cv2_compat.error):
            cv2_compat.undistort(img, K, d, newCameraMatrix=Knew)


# ---------------------------------------------------------------- scenes with lenses
K_FE = np.array([[560.0, 0.0, 615.0], [0.0, 558.0, 186.5], [0.0, 0.0, 1.0]])
D_FE = [0.02, 0.01, -0.003, 0.0002]
K_FE_WIDE = np.array([[420.0, 0.0, 620.3], [0.0, 418.0, 187.7], [0.0, 0.0, 1.0]])
SLOT = (376, 1242)


def _scaled(K, f, dc=(0.0, 0.0)):
    K = np.array(K, np.float64)
    K[0, 0] *= f
    K[1, 1] *= f
    K[0, 2] += dc[0]
    K[1, 2] += dc[1]
    return K


def lens_specs():
    """(render camera K = the sequence's camera, frame size, model, coefficients or None, raw camera or None) of six
    sequences: no lens, pinhole at its own K, pinhole with a new camera, fisheye with Knew = K, fisheye with a balance Knew,
    and a pinhole lens without coefficients whose raw camera differs from K"""
    Kb = L.fisheye_knew(cv2, K_FE_WIDE, D_FE, 376, 1241, 0.3)
    return [
        (synth.K_KITTI, (376, 1241), "pinhole", None, None),
        (_scaled(synth.K_KITTI, 1.0, (2.5, -1.0)), (375, 1240), "pinhole", U.MODELS["kitti_like_5"], None),
        (synth.K_KITTI, (370, 1226), "pinhole", [-0.05, 0.02, 0.0002, 0.0001, 0.0, 0.01, 0.004, 0.001], _scaled(synth.K_KITTI, 1.04, (3.0, 1.5))),
        (K_FE, (376, 1242), "fisheye", D_FE, None),
        (Kb, (376, 1241), "fisheye", D_FE, K_FE_WIDE),
        (synth.K_KITTI, (360, 1200), "pinhole", None, _scaled(synth.K_KITTI, 0.95, (-4.0, 2.0))),
    ]


def _raw_map(K, size, model, d, Kraw):
    """where each raw pixel of the lens (Kraw, d) lies in the image of the pinhole camera K: the map that turns a rendered
    frame into raw camera output"""
    rows, cols = size
    Kraw = K if Kraw is None else Kraw
    uv = np.stack(np.meshgrid(np.arange(cols, dtype=np.float64), np.arange(rows, dtype=np.float64)), -1).reshape(-1, 1, 2)
    if model == "fisheye":
        p = cv2.fisheye.undistortPoints(uv, Kraw, np.asarray(d, np.float64), P=K)
    else:
        p = cv2.undistortPoints(uv, Kraw, U.dist8(d)[:8], P=K)
    p = np.nan_to_num(p.reshape(rows, cols, 2), nan=-1e4, posinf=-1e4, neginf=-1e4).astype(np.float32)
    return p[..., 0], p[..., 1]


def _oracle_undistort(img, K, model, d, Kraw):
    Kraw = K if Kraw is None else Kraw
    if model == "fisheye":
        return L.fisheye_undistort(img, Kraw, d, K)
    return L.undistort_new(img, Kraw, U.dist8(d), K)


def lens_scenes(n_frames, seed0):
    out = []
    for i, (K, size, model, d, Kraw) in enumerate(lens_specs()):
        s = synth.render_sequence("kitti", n_frames, seed=seed0 + i, width=size[1], height=size[0], K=K)
        if model == "pinhole" and d is None and Kraw is None:
            raw = und = list(s["frames"])
        else:
            mx, my = _raw_map(K, size, model, d, Kraw)
            raw = [cv2.remap(f, mx, my, cv2.INTER_LINEAR, borderMode=cv2.BORDER_REFLECT_101) for f in s["frames"]]
            und = [_oracle_undistort(f, K, model, d, Kraw) for f in raw]
        coeffs = np.zeros(8)
        if d is not None:
            coeffs[:len(d)] = d
        out.append(dict(s=s, K=K, size=size, model=model, d8=coeffs, raw_K=Kraw, raw=raw, und=und))
    return out


def _lens_args(scenes):
    """set_distortion's arguments for every sequence of the scenes (one mixed call)"""
    Ks = np.stack([sc["K"] for sc in scenes])
    raw_K = np.stack([sc["K"] if sc["raw_K"] is None else sc["raw_K"] for sc in scenes])
    return np.stack([sc["d8"] for sc in scenes]), [sc["model"] for sc in scenes], raw_K, Ks


# ---------------------------------------------------------------- SequenceBatch
def test_sequence_batch_lenses_equal_undistorted_input():
    """the six lens kinds at mixed sizes against a batch without lenses fed the oracle-undistorted frames with K = the new
    camera: host steps, submitted frames and good_features"""
    n_steps = 4
    scenes = lens_scenes(n_steps + 1, 60)
    n = len(scenes)
    d8, models, raw_K, Ks = _lens_args(scenes)
    sizes = [sc["size"] for sc in scenes]
    Lm = 400
    pts = np.zeros((n, Lm, 2), np.float32)
    obj = np.zeros((n, Lm, 3), np.float32)
    n_lm = np.zeros(n, np.int32)
    for k, sc in enumerate(scenes):
        s = sc["s"]
        p = synth.grid_corners(sc["und"][0], Lm, seed=k).astype(np.float32)[:Lm]
        o = synth.backproject(sc["K"], s["R_cw"][0], s["c"][0], p.astype(np.float64), s["depth"][0]).astype(np.float32)
        pts[k, :len(p)], obj[k, :len(p)], n_lm[k] = p, o, len(p)
    a = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, dist_coeffs=d8, dist_model=models, raw_K=raw_K, max_landmarks=Lm,
                      max_candidates=Lm)
    b = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, max_landmarks=Lm, max_candidates=Lm)
    assert list(a.dist_model) == models and np.array_equal(a.dist_coeffs, d8) and np.array_equal(a.raw_K, raw_K)

    def same_features():
        ca, na = a.good_features(1400, 0.1, 10.0)
        cb, nb = b.good_features(1400, 0.1, 10.0)
        assert np.array_equal(na, nb) and np.array_equal(ca, cb)

    a.prime([sc["raw"][0] for sc in scenes])
    b.prime([sc["und"][0] for sc in scenes])
    same_features()
    ok = 0
    for t in range(1, n_steps + 1):
        if t % 2:
            ra = {k: v.copy() for k, v in a.step([sc["raw"][t] for sc in scenes], pts, obj, n_lm, pts, n_lm).items()}
            rb = b.step([sc["und"][t] for sc in scenes], pts, obj, n_lm, pts, n_lm)
        else:
            a.submit_frames([sc["raw"][t] for sc in scenes])
            b.submit_frames([sc["und"][t] for sc in scenes])
            ra = {k: v.copy() for k, v in a.step(None, pts, obj, n_lm, pts, n_lm).items()}
            rb = b.step(None, pts, obj, n_lm, pts, n_lm)
        for key in ("lm_next", "lm_status", "cand_next", "cand_status", "pose", "pnp_ok", "inlier_mask", "n_inliers"):
            assert np.array_equal(ra[key], rb[key], equal_nan=True), key
        ok += int(ra["pnp_ok"].sum())
        same_features()
    assert ok >= n * n_steps - 2, "too few poses for the comparison to mean much"
    a.close()
    b.close()


def test_set_intrinsics_keeps_an_explicit_raw_camera():
    """set_intrinsics changes only the new-camera side of a map: a batch given raw cameras and then new K equals one built
    with the new K and the same lenses; without raw_K the new K is the raw camera too"""
    scenes = lens_scenes(2, 90)
    n = len(scenes)
    d8, models, raw_K, Ks = _lens_args(scenes)
    sizes = [sc["size"] for sc in scenes]
    K2 = np.stack([_scaled(K, 1.02, (1.5, -0.5)) for K in Ks])
    frames = [sc["raw"][0] for sc in scenes]

    def features(K0, raw, K_after=None):
        x = SequenceBatch(n, *SLOT, K0, frame_size=sizes, max_landmarks=64, max_candidates=64)
        x.set_distortion(np.arange(n), d8, models, raw)
        if K_after is not None:
            x.set_intrinsics(np.arange(n), K_after)
            assert np.array_equal(x.raw_K, np.full((n, 3, 3), np.nan) if raw is None else raw, equal_nan=True)
        x.prime(frames)
        out = x.good_features(2000, 0.01, 7.0)
        x.close()
        return out

    kept, built = features(Ks, raw_K, K2), features(K2, raw_K)
    assert np.array_equal(kept[0], built[0]) and np.array_equal(kept[1], built[1])
    follows, built_none = features(Ks, None, K2), features(K2, None)
    assert np.array_equal(follows[0], built_none[0]) and np.array_equal(follows[1], built_none[1])
    assert all(not np.array_equal(kept[0][s], follows[0][s]) for s in range(n)), "the raw camera must stay what set_distortion gave"


def test_pinhole_lens_without_raw_K_is_set_distortion():
    """set_distortion(model="pinhole", raw_K=None) and raw_K = K give what b200vo_batch_set_distortion gives"""
    scenes = lens_scenes(3, 120)[:3]
    n = len(scenes)
    Ks = np.stack([sc["K"] for sc in scenes])
    sizes = [sc["size"] for sc in scenes]
    d8 = np.array([U.dist8(U.MODELS[m]) for m in ("kitti_like_5", "plumb_4", "rational_8")])
    seqs = np.arange(n, dtype=np.int32)
    out = []
    for how in ("old_abi", "none", "K"):
        x = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, max_landmarks=64, max_candidates=64)
        if how == "old_abi":
            x._call("set_distortion", n, seqs.ctypes.data_as(c_i32p), np.ascontiguousarray(d8).ctypes.data_as(c_f64p))
        else:
            x.set_distortion(seqs, d8, "pinhole", None if how == "none" else Ks)
        x.prime([sc["raw"][0] for sc in scenes])
        out.append(x.good_features(2000, 0.01, 7.0))
        x.close()
    for c, nc in out[1:]:
        assert np.array_equal(c, out[0][0]) and np.array_equal(nc, out[0][1])


# ---------------------------------------------------------------- VOBatch
CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
N_FRAMES = 14
# after the bootstrap on frames 0 and 2: full and listed steps, a reload of sequence 4 with load(K=), more steps
SCHEDULE = ([("full", None)] * 3 + [("listed", [4, 1, 0]), ("listed", [2, 3, 5]), ("listed", [5, 0, 3])] + [("full", None)] * 2
            + [("load", 4), ("load", 2)] + [("full", None)] * 3 + [("listed", [0, 1, 2, 3, 4, 5])])


@pytest.fixture(scope="module")
def scenes():
    return lens_scenes(N_FRAMES, 800)


def _same_lenses(before, x):
    """the mirrors dist_coeffs, dist_model, raw_K equal the saved ones"""
    assert np.array_equal(before[0], x.dist_coeffs) and np.array_equal(before[1], x.dist_model)
    assert np.array_equal(before[2], x.raw_K, equal_nan=True)


def _refusals(vb, n):
    """every bad set_distortion raises and changes nothing"""
    before = (vb.dist_coeffs.copy(), vb.dist_model.copy(), vb.raw_K.copy())
    status = [vb.read_state(s)["status"] for s in range(n)]
    fe, K = np.array(D_FE), K_FE
    skew = K.copy()
    skew[0, 1] = 0.1
    for args in ((([0, 0], [fe, fe], "fisheye", None)), (([6], [fe], "fisheye", None)),
                 (([0], [fe], "bogus", None)), (([0, 1], [fe, fe], ["fisheye"] * 3, None)), (([0], [fe[:3]], "fisheye", None)),
                 (([0], [np.r_[fe, 0.0]], "fisheye", None)), (([0, 1], [np.r_[fe, 0.1], np.zeros(5)], ["fisheye", "pinhole"], None)),
                 (([0], [[np.nan, 0, 0, 0]], "fisheye", None)), (([0], [fe], "fisheye", K)), (([0], [fe], "fisheye", skew[None])),
                 (([0], [fe], "fisheye", np.diag([np.nan, 1.0, 1.0])[None])), (([0], [fe], "fisheye", np.diag([-1.0, 1.0, 1.0])[None])),
                 (([0], np.zeros((1, 6)), "pinhole", None)), (([0], np.zeros((1, 3)), "pinhole", None))):
        seqs, d, model, raw = args
        with pytest.raises(ValueError):
            vb.set_distortion(seqs, d, model, raw)
    with pytest.raises(NotImplementedError):
        vb.set_distortion([0], np.zeros((1, 12)))
    code = np.int32([7])
    with pytest.raises(ValueError):   # an unknown model code at the C ABI
        vb._call("set_lens", 1, np.int32([0]).ctypes.data_as(c_i32p), code.ctypes.data_as(c_i32p),
                 np.zeros(8).ctypes.data_as(c_f64p), None)
    _same_lenses(before, vb)
    assert [vb.read_state(s)["status"] for s in range(n)] == status


def _run(scenes, lens):
    """One VOBatch of the scenes following SCHEDULE.  lens: the sequences get raw frames and their lenses; otherwise every
    sequence gets the oracle-undistorted frames.  -> (bootstrap result, per sequence the (result row, state) of every advance)"""
    n = len(scenes)
    d8, models, raw_K, Ks = _lens_args(scenes)
    vb = VOBatch(n, *SLOT, Ks, OPT, frame_size=[sc["size"] for sc in scenes], **CAPS)
    key = "raw" if lens else "und"
    if lens:
        _refusals(vb, n)
        vb.set_distortion(np.arange(n), d8, models, raw_K)
        assert all(vb.read_state(s)["status"] == VOBatch.IDLE for s in range(n))
        _refusals(vb, n)
    boot = {k: np.array(v) for k, v in vb.bootstrap([sc[key][0] for sc in scenes], [sc[key][2] for sc in scenes], K=Ks).items()}
    if lens:
        assert np.array_equal(vb.raw_K, raw_K)
    nxt = [3] * n
    log = [[(None, vb.read_state(s))] for s in range(n)]
    for form, arg in SCHEDULE:
        if form == "load":
            st = vb.read_state(arg)
            vb.load(arg, scenes[arg][key][nxt[arg] - 1], st, K=Ks[arg])
            log[arg].append((None, vb.read_state(arg)))
            continue
        listed = list(range(n)) if arg is None else arg
        images = [scenes[s][key][nxt[s]] for s in listed]
        r = {k: np.array(v) for k, v in (vb.step(images) if arg is None else vb.step(images, seqs=arg)).items()}
        for row, s in enumerate(listed):
            log[s].append(({k: r[k][row].copy() for k in r}, vb.read_state(s)))
            nxt[s] += 1
    if lens:
        assert np.array_equal(vb.raw_K, raw_K) and list(vb.dist_model) == models
    vb.close()
    return boot, log


def test_vobatch_lenses(scenes):
    boot, log = _run(scenes, True)
    ref_boot, ref_log = _run(scenes, False)
    oks = 0
    for s in range(len(scenes)):
        for k in boot:
            assert boot[k][s] == ref_boot[k][s], (s, k)
        assert boot["status"][s] == VOBatch.OK, s
        assert len(log[s]) == len(ref_log[s])
        for (ra, sa), (rb, sb) in zip(log[s], ref_log[s]):
            if ra is not None:
                for k in ra:
                    assert np.array_equal(ra[k], rb[k], equal_nan=True), (s, k)
                oks += int(ra["status"] == VOBatch.OK)
            for k in STATE_KEYS:
                assert np.array_equal(sa[k], sb[k], equal_nan=True), (s, k)
            assert sa["status"] == sb["status"], s
    n_adv = sum(ra is not None for s in range(len(scenes)) for ra, _ in log[s])
    assert oks >= 0.8 * n_adv, f"only {oks} of {n_adv} steps stayed OK: the comparison would mean little"


def test_lens_refused_while_submitted_frames_wait(scenes):
    """a new lens, and a K of a sequence with a map, are refused while a submitted set waits; nothing changes"""
    n = len(scenes)
    d8, models, raw_K, Ks = _lens_args(scenes)
    sb = SequenceBatch(n, *SLOT, Ks, frame_size=[sc["size"] for sc in scenes], dist_coeffs=d8, dist_model=models, raw_K=raw_K,
                       max_landmarks=64, max_candidates=64)
    sb.prime([sc["raw"][0] for sc in scenes])
    sb.submit_frames([sc["raw"][1] for sc in scenes])
    before = (sb.dist_coeffs.copy(), sb.dist_model.copy(), sb.raw_K.copy())
    with pytest.raises(ValueError):
        sb.set_distortion([0], [D_FE], "fisheye")
    for s in (3, 4, 5):   # fisheye, fisheye with a raw camera, a raw camera alone
        with pytest.raises(ValueError):
            sb.set_intrinsics([s], _scaled(Ks[s], 1.01)[None])
    sb.set_intrinsics([0], Ks[0][None])   # a sequence without a map keeps today's behaviour
    _same_lenses(before, sb)
    sb.close()
