"""Detection masks on the device: the per-call masked forms (cv2_compat.good_features_to_track_masked,
sift_detect_and_compute(mask=)) against tests/mask_reference.py and cv2, and the per-sequence masks of SequenceBatch / VOBatch
(set_detection_mask): a masked sequence computes exactly what the per-call masked forms compute on its frames, an unmasked
one exactly what it computes in a batch without masks."""
import numpy as np
import pytest

import mask_reference as R
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT, rodrigues
from monocular_visual_odometry_va4mr_b200 import cv2_compat, hotpath, synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch, initial_state, match_bootstrap_frames

pytestmark = pytest.mark.gpu

CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
SLOT = (376, 1242)
N_FRAMES = 25
GFTT_ARGS = (OPT["feature_max_corners"], OPT["feature_quality_level"], OPT["feature_min_dist"])


def _K(fx, fy, cx, cy):
    return np.array([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]])


KITTI = [(_K(718.856, 718.856, 607.1928, 185.2157), (376, 1241)), (_K(721.5377, 721.5377, 609.5593, 172.854), (375, 1242)),
         (_K(707.0912, 707.0912, 601.8873, 183.1104), (370, 1226))]


def _same(a, b):
    if a is None or b is None:
        return a is None and b is None
    return a.shape == b.shape and np.array_equal(a, b)


# ---------------------------------------------------------------- per-call forms
@pytest.fixture(scope="module")
def frames():
    return [synth.render_sequence("kitti", 1, seed=s)["frames"][0] for s in (0, 7)]


def test_gftt_masked_per_call(frames):
    import cv2
    for k, img in enumerate(frames):
        for name, mask in R.standard_masks(img, seed=k).items():
            got = cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, mask)
            assert _same(got, R.good_features_to_track(img, *GFTT_ARGS, mask=mask)), (k, name)
            assert _same(got, cv2.goodFeaturesToTrack(img, *GFTT_ARGS, mask=mask, blockSize=3)), (k, name)
        for x, y in cv2_compat.goodFeaturesToTrack(img, *GFTT_ARGS).reshape(-1, 2)[:3].astype(int):   # one pixel on a corner
            one = np.zeros(img.shape, np.uint8)
            one[y, x] = 255
            assert np.array_equal(cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, one).reshape(-1, 2), [[x, y]])
        # no mask: the unmasked entry, bit for bit
        assert _same(cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, None), cv2_compat.goodFeaturesToTrack(img, *GFTT_ARGS))


def test_gftt_masked_per_call_negative_eigenvalues():
    for img, one, nine in R.negative_eig_cases():
        for m in (one, nine):
            for q in (0.01, 0.1, 1.0):
                assert cv2_compat.good_features_to_track_masked(img, 10, q, 1, m) is None


def test_gftt_masked_per_call_bitonic_path():
    img = R.checkerboard()
    for name, mask in R.standard_masks(img).items():
        got = cv2_compat.good_features_to_track_masked(img, 0, 0.5, 0, mask)
        assert _same(got, R.good_features_to_track(img, 0, 0.5, 0, mask=mask)), name
    assert len(cv2_compat.good_features_to_track_masked(img, 0, 0.5, 0, R.hood_mask(img.shape))) > 32768


def test_per_call_mask_refusals(frames):
    img = frames[0]
    for bad in (np.zeros((10, 10), np.uint8), np.zeros(img.shape, np.float32), np.zeros(img.shape + (1,), np.uint8), [[1]]):
        with pytest.raises(cv2_compat.error):
            cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, bad)
        with pytest.raises(cv2_compat.error):
            cv2_compat.sift_detect_and_compute(img, mask=bad)
    # the drop-in names keep refusing mask=
    with pytest.raises(NotImplementedError):
        cv2_compat.goodFeaturesToTrack(img, *GFTT_ARGS, mask=np.ones(img.shape, np.uint8))
    with pytest.raises(NotImplementedError):
        cv2_compat.SIFT_create().detectAndCompute(img, np.ones(img.shape, np.uint8))


@pytest.mark.parametrize("seed", [0, 3])
def test_sift_masked_per_call(seed):
    img = synth.render_sequence("kitti", 1, seed=seed)["frames"][0]
    kp0, oc0, d0 = cv2_compat.sift_detect_and_compute(img)
    masks = {k: v for k, v in R.standard_masks(img).items() if k in ("hood", "wedges", "blobs", "all_7", "all_0")}
    edge = np.full(img.shape, 255, np.uint8)           # zero bytes where the keypoints closest to x.5 / y.5 round to
    frac = np.abs(kp0[:, :2] % 1 - 0.5).min(axis=1)
    for x, y in kp0[np.argsort(frac)[:40], :2]:
        edge[int(np.float32(y) + np.float32(0.5)), int(np.float32(x) + np.float32(0.5))] = 0
    masks["half_pixel_edges"] = edge
    for name, mask in masks.items():
        kp, oc, d = cv2_compat.sift_detect_and_compute(img, mask=mask)
        rk, ro, rd = R.sift_detect_and_compute(img, mask)
        assert np.array_equal(kp, rk) and np.array_equal(oc, ro) and np.array_equal(d, rd), name
        keep = R.sift_mask_keep(kp0[:, :2], mask)
        assert np.array_equal(kp, kp0[keep]) and np.array_equal(d, d0[keep]), name
    kp, oc, d = cv2_compat.sift_detect_and_compute(img, mask=None)
    assert np.array_equal(kp, kp0) and np.array_equal(oc, oc0) and np.array_equal(d, d0)


# ---------------------------------------------------------------- SequenceBatch.good_features
def test_sequence_batch_good_features_with_masks():
    sizes = [KITTI[0][1], KITTI[1][1], KITTI[2][1], KITTI[0][1], (300, 1000)]
    imgs = [synth.render_sequence("kitti", 1, seed=40 + i, width=c, height=r)["frames"][0] for i, (r, c) in enumerate(sizes)]
    masks = {0: R.hood_mask(sizes[0]), 2: R.wedge_mask(sizes[2]), 4: R.blob_mask(sizes[4], 3)}
    sb = SequenceBatch(len(sizes), *SLOT, KITTI[0][0], frame_size=sizes)
    sb.prime(imgs)
    plain_c, plain_n = sb.good_features(*GFTT_ARGS)
    seqs = sorted(masks)
    sb.set_detection_mask(seqs, [masks[s] for s in seqs])
    assert list(np.flatnonzero(sb.has_mask)) == seqs
    c, n = sb.good_features(*GFTT_ARGS)
    for s, img in enumerate(imgs):
        want = cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, masks.get(s))
        assert n[s] == len(want) and np.array_equal(c[s, :n[s]], want.reshape(-1, 2)), s
        if s not in masks:
            assert n[s] == plain_n[s] and np.array_equal(c[s], plain_c[s])
    # set_frame_size clears the listed sequences' masks; None clears them too
    sb.set_frame_size([0], [sizes[0]])
    assert not sb.has_mask[0]
    sb.prime(imgs)
    c, n = sb.good_features(*GFTT_ARGS)
    assert n[0] == plain_n[0] and np.array_equal(c[0], plain_c[0])
    assert n[2] != plain_n[2] or not np.array_equal(c[2], plain_c[2])
    sb.set_detection_mask([2, 4], None)
    c, n = sb.good_features(*GFTT_ARGS)
    assert np.array_equal(n, plain_n) and np.array_equal(c, plain_c)
    sb.close()


def test_sequence_batch_masked_maximum():
    """The batched detector's masked maximum (gftt_mask_max_kernel): a quiet patch alone, the same patch with the 1-pixel
    border ring setting the threshold, and one image masked on its border ring alone, at mixed frame sizes."""
    sizes = [KITTI[0][1], KITTI[2][1], (300, 1000)]
    imgs = [synth.render_sequence("kitti", 1, seed=60 + i, width=c, height=r)["frames"][0] for i, (r, c) in enumerate(sizes)]
    pm = [R.patch_masks(img) for img in imgs]
    ring_only = pm[2]["patch_and_ring"].copy()
    ring_only[ring_only == 255] = 0
    masks = [pm[0]["quiet_patch"], pm[1]["patch_and_ring"], ring_only]
    sb = SequenceBatch(len(sizes), *SLOT, KITTI[0][0], frame_size=sizes)
    sb.prime(imgs)
    sb.set_detection_mask(range(len(sizes)), masks)
    c, n = sb.good_features(*GFTT_ARGS)
    for s, img in enumerate(imgs):
        want = R.good_features_to_track(img, *GFTT_ARGS, mask=masks[s])
        got = cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, masks[s])
        assert _same(got, want), s
        assert n[s] == (0 if want is None else len(want)), s
        if want is not None:
            assert np.array_equal(c[s, :n[s]], want.reshape(-1, 2)), s
    # the ring raises the threshold above the patch's own maximum: fewer corners than the patch alone gives
    alone = R.good_features_to_track(imgs[1], *GFTT_ARGS, mask=pm[1]["quiet_patch"])
    assert alone is not None and n[1] < len(alone)
    assert n[2] == 0                          # no interior pixel in the mask: no corner
    sb.close()


def test_sequence_batch_negative_masked_maximum():
    """One-pixel and 3 x 3 masks on pixels of negative eigenvalue: the batched detector's masked maximum is clamped at 0
    and finds nothing, as cv2 does, while the unmasked sequences of the batch keep their corners."""
    cases = R.negative_eig_cases()
    imgs = [img for img, _, _ in cases]
    h, w = imgs[0].shape
    sb = SequenceBatch(2 * len(cases) + 1, h, w, KITTI[0][0], win=(7, 7), max_level=1)
    sb.prime(imgs + imgs + [imgs[0]])
    sb.set_detection_mask(range(2 * len(cases)), [one for _, one, _ in cases] + [nine for _, _, nine in cases])
    for q in (0.01, 0.1, 1.0):
        c, n = sb.good_features(10, q, 1.0)
        assert (n[:-1] == 0).all(), (q, n)
        want = cv2_compat.goodFeaturesToTrack(imgs[0], 10, q, 1.0)
        assert n[-1] == (0 if want is None else len(want)), q
        if want is not None:
            assert np.array_equal(c[-1, :n[-1]], want.reshape(-1, 2)), q
    sb.close()


# ---------------------------------------------------------------- VOBatch
@pytest.fixture(scope="module")
def scenes():
    """Six sequences, two per KITTI group at its size and calibration; every other one with a detection mask."""
    kinds = [R.hood_mask, R.wedge_mask, lambda shape: R.blob_mask(shape, 5)]
    out = []
    for i in range(6):
        K, (r, c) = KITTI[i // 2]
        s = synth.render_sequence("kitti", N_FRAMES, seed=500 + i, width=c, height=r, K=K)
        mask = kinds[i // 2]((r, c)) if i % 2 == 0 else None
        out.append((s["frames"], K, (r, c), mask))
    return out


MASKED = [0, 2, 4]


def _percall_step(st, prev, img, K, pose_cw, mask):
    """MiniVO.step on the per-call entry points with the masked detector (the loop test's _percall_step otherwise)."""
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
    c = cv2_compat.good_features_to_track_masked(img, *GFTT_ARGS, mask, blockSize=o["feature_block_size"])
    c = np.zeros((0, 2), np.float32) if c is None else c.reshape(-1, 2)
    c = c[hotpath.min_distance_mask(c, keys, o["feature_min_dist"])]
    new = dict(lm=lm, lm_kp=kp, keys=np.concatenate([keys, c]), first_keys=np.concatenate([fk, c]),
               first_pose=np.concatenate([fp, np.full(len(c), len(poses), np.int32)]), poses=np.vstack([poses, pose_cw]))
    return VOBatch.OK, len(inl), host, new


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def _slot(images):
    out = np.zeros((len(images),) + SLOT, np.uint8)
    for k, im in enumerate(images):
        out[k, :im.shape[0], :im.shape[1]] = im
    return out


# the schedule after the bootstrap on frames 0 and 2: (form, listed sequences or None); every sequence advances one frame
# when it is listed.  Full steps, listed steps, step_dev with frames submitted ahead, and full steps after the masks are
# cleared ("clear" marks the point).
SCHEDULE = ([("full", None)] * 6 + [("listed", [4, 1, 0]), ("listed", [2, 3, 5]), ("listed", [5, 0]), ("listed", [1, 2, 3, 4])]
            + [("dev", None)] * 6 + [("listed", [0, 1, 2, 3, 4, 5])] + [("clear", None)] + [("full", None)] * 3)


def _refusals(vb, scenes):
    """every bad set_detection_mask raises ValueError and changes nothing"""
    good = [scenes[s][3] for s in MASKED]
    before = vb.has_mask.copy()
    for seqs, masks in (([0, 0], good[:2]), ([6], good[:1]), ([-1], good[:1]), ([], []), ([[0]], good[:1]),
                        ([0, 2], good), ([0], [good[0][:-1]]), ([0], [good[0].astype(np.int16)]),
                        ([0, 2], np.zeros((2, 10, 10), np.uint8)), ([0], np.zeros((1,) + SLOT, np.float32))):
        with pytest.raises(ValueError):
            vb.set_detection_mask(seqs, masks)
    with pytest.raises(ValueError):
        vb.set_detection_mask([0, 0], None)
    assert np.array_equal(vb.has_mask, before)


def _run(scenes, masked, check=None):
    """One VOBatch of the scenes following SCHEDULE; masked: set the scenes' masks.  -> per sequence, per advance:
    (result row, state).  check(s, prev_f, f, row, state, mask): the per-call comparison, or None."""
    import torch
    vb = VOBatch(len(scenes), *SLOT, np.stack([K for _, K, _, _ in scenes]), OPT, frame_size=[sz for _, _, sz, _ in scenes], **CAPS)
    n = len(scenes)
    if masked:
        _refusals(vb, scenes)
        vb.set_detection_mask(MASKED, [scenes[s][3] for s in MASKED])
        assert list(np.flatnonzero(vb.has_mask)) == MASKED
        _refusals(vb, scenes)
    masks = [scenes[s][3] if masked else None for s in range(n)]
    boot = {k: np.array(v) for k, v in vb.bootstrap([fr[0] for fr, *_ in scenes], [fr[2] for fr, *_ in scenes]).items()}
    nxt = [3] * n
    log = [[(None, vb.read_state(s))] for s in range(n)]
    dev_frames = []
    z = lambda *shape, dt=torch.int32: torch.zeros(shape, dtype=dt, device="cuda")
    out = dict(status=z(n), n_inliers=z(n), n_lm=z(n), n_cand=z(n), pose_cw=z(n, 12, dt=torch.float64))
    for form, seqs in SCHEDULE:
        if form == "clear":
            if masked:
                vb.set_detection_mask(MASKED, None)
                assert not vb.has_mask.any()
            masks = [None] * n
            continue
        listed = list(range(n)) if seqs is None else seqs
        images = [scenes[s][0][nxt[s]] for s in listed]
        if form == "full":
            r = {k: np.array(v) for k, v in vb.step(images).items()}
        elif form == "listed":
            r = {k: np.array(v) for k, v in vb.step(images, seqs=seqs).items()}
        else:
            f = torch.from_numpy(_slot(images)).cuda()
            torch.cuda.synchronize()
            dev_frames.append(f)
            vb.submit_frames_dev(f.data_ptr())
            vb.step_dev(None, {k: v.data_ptr() for k, v in out.items()})
            vb.ctx.sync()
            r = {k: v.cpu().numpy() for k, v in out.items()}
        for row, s in enumerate(listed):
            res = {k: r[k][row].copy() for k in r}
            st = vb.read_state(s)
            if check is not None:
                check(s, nxt[s] - 1, nxt[s], res, st, masks[s])
            log[s].append((res, st))
            nxt[s] += 1
    vb.close()
    return boot, log


def test_vobatch_masks(scenes):
    """Masked and unmasked sequences of three sizes and cameras, 20+ steps in every form: each sequence equals MiniVO on the
    per-call entries with its own mask (bootstrap: the host chain with match_bootstrap_frames(mask=)), and each unmasked one
    equals the same batch run without masks."""
    ref, live = {}, {}

    def check(s, pf, f, res, st, mask):
        frames, K, _, _ = scenes[s]
        if not live[s]:
            assert res["status"] != VOBatch.OK
            return
        code, n_inl, host, new = _percall_step(ref[s], frames[pf], frames[f], K, res["pose_cw"].copy(), mask)
        assert res["status"] == code and res["n_inliers"] == n_inl, (s, f)
        if code != VOBatch.OK:
            live[s] = False
            return
        assert np.abs(res["pose_cw"] - host).max() <= 1e-12, (s, f)
        assert res["n_lm"] == len(new["lm"]) and res["n_cand"] == len(new["keys"]), (s, f)
        _assert_state(st, new)
        ref[s] = new

    for s, (frames, K, _, mask) in enumerate(scenes):
        st = initial_state(K, OPT, *match_bootstrap_frames(frames[0], frames[2], OPT["feature_ratio"], mask=mask))
        ref[s] = {k: st[k] for k in STATE_KEYS}
        ref[s]["num_pts"] = st["num_pts"]
        live[s] = True
    boot_ref = {s: dict(ref[s]) for s in ref}
    boot, log = _run(scenes, True, check)
    for s in range(len(scenes)):
        assert boot["status"][s] == VOBatch.OK and boot["num_pts"][s] == boot_ref[s]["num_pts"], s
        _assert_state(log[s][0][1], boot_ref[s])
    assert sum(live.values()) >= 4, "too few sequences stayed live for the comparison to mean much"
    # the masks changed what the masked sequences detect
    plain_boot, plain_log = _run(scenes, False)
    for s in range(len(scenes)):
        if s in MASKED:
            assert any(a[1]["keys"].shape != b[1]["keys"].shape or not np.array_equal(a[1]["keys"], b[1]["keys"])
                       for a, b in zip(log[s], plain_log[s])), s
            continue
        for k in boot:
            assert boot[k][s] == plain_boot[k][s], (s, k)
        for (ra, sa), (rb, sb) in zip(log[s], plain_log[s]):
            if ra is not None:
                for k in ra:
                    assert np.array_equal(ra[k], rb[k]), (s, k)
            _assert_state(sa, sb)
            assert sa["status"] == sb["status"]


def test_vobatch_set_frame_size_clears_masks(scenes):
    frames, K, size, mask = scenes[0]
    vb = VOBatch(2, *SLOT, K, OPT, frame_size=[size, size], **CAPS)
    vb.set_detection_mask([0, 1], [mask, mask])
    vb.set_frame_size([1], [size])
    assert list(vb.has_mask) == [True, False]
    boot = vb.bootstrap([frames[0]] * 2, [frames[2]] * 2)
    st = [vb.read_state(s) for s in range(2)]
    want = initial_state(K, OPT, *match_bootstrap_frames(frames[0], frames[2], OPT["feature_ratio"]))
    assert boot["num_pts"][1] == want["num_pts"]
    _assert_state(st[1], want)
    vb.close()
