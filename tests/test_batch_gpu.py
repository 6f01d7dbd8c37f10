"""Batched KLT + PnP step (b200vo_batch_step) against the per-call path, the oracle and live cv2."""
import numpy as np
import pytest

from monocular_visual_odometry_va4mr_b200 import cv2_compat, workload
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def wl():
    return workload.TrackWorkload("kitti", batch=5, n_frames=3, n_landmarks=300, n_candidates=200, n_distinct=2,
                                  seed=1, width=640, height=240, cap_landmarks=320, cap_candidates=256)


def _run_steps(wl, n_steps, opts, pinned=False):
    sb = SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                       pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                       max_landmarks=wl.L, max_candidates=wl.Cn)
    order = workload.frame_order(wl.F, n_steps)
    frames = wl.frames
    if pinned:
        frames = sb.pinned_frames(wl.F)
        frames[:] = wl.frames
    sb.prime(frames[order[0]])
    outs = []
    for t in range(n_steps):
        f, g = order[t], order[t + 1]
        o = sb.step(frames[g], wl.lm_pts[f], wl.lm_obj[f], wl.n_lm[f], wl.cand_pts[f], wl.n_cand[f])
        outs.append({k: v.copy() for k, v in o.items()})
    sb.close()
    return order, outs


@pytest.mark.parametrize("pinned", [False, True])
def test_batch_equals_per_call_path(wl, pinned):
    opts = workload.REFERENCE_OPTIONS["kitti"]
    order, outs = _run_steps(wl, 4, opts, pinned)
    for t, o in enumerate(outs):
        f, g = order[t], order[t + 1]
        for s in range(wl.batch):
            nl, nc = int(wl.n_lm[f, s]), int(wl.n_cand[f, s])
            p, st, _ = cv2_compat.calcOpticalFlowPyrLK(wl.frames[f, s], wl.frames[g, s], wl.lm_pts[f, s, :nl], None,
                                                       winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
            assert np.array_equal(o["lm_status"][s, :nl], st.ravel())
            assert np.array_equal(o["lm_next"][s, :nl], p)
            pc, stc, _ = cv2_compat.calcOpticalFlowPyrLK(wl.frames[f, s], wl.frames[g, s], wl.cand_pts[f, s, :nc], None,
                                                         winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
            assert np.array_equal(o["cand_status"][s, :nc], stc.ravel())
            assert np.array_equal(o["cand_next"][s, :nc], pc)
            keep = st.ravel() == 1
            ok, rv, tv, inl = cv2_compat.solvePnPRansac(wl.lm_obj[f, s, :nl][keep], p[keep], wl.K, np.zeros(4),
                                                        flags=cv2_compat.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                                                        reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
            assert bool(o["pnp_ok"][s]) == ok
            mask = np.zeros(wl.L, np.uint8)
            mask[np.flatnonzero(keep)[inl.ravel()]] = 1
            assert np.array_equal(o["inlier_mask"][s], mask)
            assert int(o["n_inliers"][s]) == len(inl)
            assert np.array_equal(o["pose"][s], np.concatenate([rv.ravel(), tv.ravel()]))


def test_unfused_pose_path_equals_fused(wl):
    """A landmark capacity above VO_PNP_FUSED_MAX_N (4096, csrc/pnp.cuh) runs the separate pose kernels (status compaction,
    RANSAC, select, EPnP, mask scatter) instead of the fused one.  Against a twin at capacity 4096 stepped on the same data:
    identical tracks, decisions and inliers; poses to rounding, since the two paths run different 12x12 Jacobi schedules."""
    opts = workload.REFERENCE_OPTIONS["kitti"]
    fused_max, n_steps = 4096, 3
    order = workload.frame_order(wl.F, n_steps)
    outs = {}
    for L in (fused_max + 4, fused_max):
        lm_pts = np.zeros((wl.F, wl.batch, L, 2), np.float32)
        lm_obj = np.zeros((wl.F, wl.batch, L, 3), np.float32)
        lm_pts[:, :, :wl.L], lm_obj[:, :, :wl.L] = wl.lm_pts, wl.lm_obj
        sb = SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                           pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                           max_landmarks=L, max_candidates=wl.Cn)
        sb.prime(wl.frames[order[0]])
        outs[L] = []
        for t in range(n_steps):
            f, g = order[t], order[t + 1]
            o = sb.step(wl.frames[g], lm_pts[f], lm_obj[f], wl.n_lm[f], wl.cand_pts[f], wl.n_cand[f])
            outs[L].append({k: v.copy() for k, v in o.items()})
        sb.close()
    for t in range(n_steps):
        u, w = outs[fused_max + 4][t], outs[fused_max][t]
        for s in range(wl.batch):
            nl = int(wl.n_lm[order[t], s])
            assert np.array_equal(u["lm_status"][s, :nl], w["lm_status"][s, :nl]), (t, s)
            assert np.array_equal(u["inlier_mask"][s, :fused_max], w["inlier_mask"][s]) and not u["inlier_mask"][s, fused_max:].any(), (t, s)
        assert u["pnp_ok"].all() and np.array_equal(u["pnp_ok"], w["pnp_ok"]) and np.array_equal(u["n_inliers"], w["n_inliers"]), t
        d = np.abs(u["pose"] - w["pose"]).max()
        assert d <= 1e-9, (t, d)


def test_batch_vs_oracle_and_truth(wl):
    import oracle
    opts = workload.REFERENCE_OPTIONS["kitti"]
    order, outs = _run_steps(wl, 2, opts)
    for t, o in enumerate(outs):
        f, g = order[t], order[t + 1]
        for s in range(wl.batch):
            nl = int(wl.n_lm[f, s])
            rp, rst, _ = oracle.calc_optical_flow_pyr_lk(wl.frames[f, s], wl.frames[g, s], wl.lm_pts[f, s, :nl],
                                                         opts["win"], opts["max_level"], opts["criteria"])
            assert np.array_equal(o["lm_status"][s, :nl], rst.ravel())
            keep = rst.ravel() == 1
            assert np.abs(o["lm_next"][s, :nl] - rp)[keep].max() <= 0.05
            ok, rv, tv, inl, _ = oracle.solve_pnp_ransac_p3p(wl.lm_obj[f, s, :nl][keep], rp[keep], wl.K, opts["pnp_iters"],
                                                             opts["pnp_err"], opts["pnp_conf"])
            assert ok and o["pnp_ok"][s]
            assert np.array_equal(np.flatnonzero(o["inlier_mask"][s]), np.flatnonzero(keep)[inl.ravel()])
            assert np.abs(o["pose"][s] - np.concatenate([rv.ravel(), tv.ravel()])).max() < 1e-6
            # and the recovered pose is the rendered camera (synthetic ground truth), loosely
            R, tt = wl.true_pose(s, g)
            assert np.abs(oracle.rodrigues_to_R(o["pose"][s, :3]) - R).max() < 0.02
            assert np.abs(o["pose"][s, 3:] - tt).max() < 0.3


def test_batch_live_cv2(wl):
    cv2 = pytest.importorskip("cv2")
    opts = workload.REFERENCE_OPTIONS["kitti"]
    order, outs = _run_steps(wl, 2, opts)
    for t, o in enumerate(outs):
        f, g = order[t], order[t + 1]
        for s in range(wl.batch):
            nl = int(wl.n_lm[f, s])
            p, st, _ = cv2.calcOpticalFlowPyrLK(wl.frames[f, s], wl.frames[g, s], wl.lm_pts[f, s, :nl], None,
                                                winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
            assert np.array_equal(o["lm_status"][s, :nl], st.ravel())
            keep = st.ravel() == 1
            d = np.abs(o["lm_next"][s, :nl] - p)[keep].max(axis=1)
            assert (d <= 0.05).mean() >= 0.99
            if d.max() == 0:   # identical tracked positions -> PnP must agree exactly on the inlier set
                ok, rv, tv, inl = cv2.solvePnPRansac(wl.lm_obj[f, s, :nl][keep], p[keep], wl.K, np.zeros(4),
                                                     flags=cv2.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                                                     reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
                assert np.array_equal(np.flatnonzero(o["inlier_mask"][s]), np.flatnonzero(keep)[inl.ravel()])


def test_prefetched_frames_equal_call_by_call(wl):
    """b200vo_batch_submit_frames(t+1) + step(frames=None) must give the bits of step(frames)."""
    opts = workload.REFERENCE_OPTIONS["kitti"]
    n_steps = 5
    order, ref = _run_steps(wl, n_steps, opts, pinned=True)
    sb = SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                       pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                       max_landmarks=wl.L, max_candidates=wl.Cn)
    frames = sb.pinned_frames(wl.F)
    frames[:] = wl.frames
    sb.prime(frames[order[0]])
    sb.submit_frames(frames[order[1]])
    for t in range(n_steps):
        f = order[t]
        if t + 2 <= n_steps:
            sb.submit_frames(frames[order[t + 2]])     # two sets waiting at most
        o = sb.step(None, wl.lm_pts[f], wl.lm_obj[f], wl.n_lm[f], wl.cand_pts[f], wl.n_cand[f])
        for k, v in o.items():
            assert np.array_equal(v, ref[t][k]), (t, k)
    # protocol errors: nothing submitted / a set is waiting but frames are passed / pageable frames
    from monocular_visual_odometry_va4mr_b200._lib import B200VOError
    with pytest.raises(B200VOError):
        sb.step(None, wl.lm_pts[0], wl.lm_obj[0], wl.n_lm[0], wl.cand_pts[0], wl.n_cand[0])
    with pytest.raises(B200VOError):
        sb.submit_frames(np.ascontiguousarray(wl.frames[0]))
    sb.submit_frames(frames[0])
    with pytest.raises(B200VOError):
        sb.step(frames[1], wl.lm_pts[0], wl.lm_obj[0], wl.n_lm[0], wl.cand_pts[0], wl.n_cand[0])
    sb.close()


@pytest.mark.parametrize("shape,w,h", [("parking", 640, 480), ("malaga", 512, 384)])
def test_batch_other_shapes_equal_per_call_path(shape, w, h):
    """The reference's Parking / Malaga options (maxLevel 10 -> 5 or 6 levels, PnP_error 5) through the batched step."""
    opts = workload.REFERENCE_OPTIONS[shape]
    wl2 = workload.TrackWorkload(shape, batch=3, n_frames=3, n_landmarks=200, n_candidates=100, n_distinct=2, seed=3,
                                 width=w, height=h, cap_landmarks=256, cap_candidates=128)
    order, outs = _run_steps(wl2, 2, opts, pinned=True)
    for t, o in enumerate(outs):
        f, g = order[t], order[t + 1]
        for s in range(wl2.batch):
            nl, nc = int(wl2.n_lm[f, s]), int(wl2.n_cand[f, s])
            p, st, _ = cv2_compat.calcOpticalFlowPyrLK(wl2.frames[f, s], wl2.frames[g, s], wl2.lm_pts[f, s, :nl], None,
                                                       winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
            assert np.array_equal(o["lm_status"][s, :nl], st.ravel()) and np.array_equal(o["lm_next"][s, :nl], p)
            if nc:
                pc, stc, _ = cv2_compat.calcOpticalFlowPyrLK(wl2.frames[f, s], wl2.frames[g, s], wl2.cand_pts[f, s, :nc], None,
                                                             winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
                assert np.array_equal(o["cand_status"][s, :nc], stc.ravel()) and np.array_equal(o["cand_next"][s, :nc], pc)
            keep = st.ravel() == 1
            if keep.sum() < 4:
                continue
            ok, rv, tv, inl = cv2_compat.solvePnPRansac(wl2.lm_obj[f, s, :nl][keep], p[keep], wl2.K, np.zeros(4),
                                                        flags=cv2_compat.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                                                        reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
            assert bool(o["pnp_ok"][s]) == ok
            if ok:
                mask = np.zeros(wl2.L, np.uint8)
                mask[np.flatnonzero(keep)[inl.ravel()]] = 1
                assert np.array_equal(o["inlier_mask"][s], mask)
                assert np.array_equal(o["pose"][s], np.concatenate([rv.ravel(), tv.ravel()]))


def test_batch_ragged_counts(wl):
    """Sequences with 0, 3, 4, 5 ... landmarks and 0 candidates in one batch: < 4 tracked landmarks -> pnp_ok 0 (the
    reference raises "Not enough keypoints" there, :360), the others equal the per-call path."""
    opts = workload.REFERENCE_OPTIONS["kitti"]
    n_lm = wl.n_lm.copy()
    n_cand = wl.n_cand.copy()
    n_lm[:, 0] = 0; n_lm[:, 1] = 3; n_lm[:, 2] = 4; n_lm[:, 3] = 5
    n_cand[:, 0] = 0; n_cand[:, 4] = 1
    sb = SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                       pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                       max_landmarks=wl.L, max_candidates=wl.Cn)
    sb.prime(wl.frames[0])
    o = sb.step(wl.frames[1], wl.lm_pts[0], wl.lm_obj[0], n_lm[0], wl.cand_pts[0], n_cand[0])
    for s in range(wl.batch):
        nl = int(n_lm[0, s])
        if nl:
            p, st, _ = cv2_compat.calcOpticalFlowPyrLK(wl.frames[0, s], wl.frames[1, s], wl.lm_pts[0, s, :nl], None,
                                                       winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
            assert np.array_equal(o["lm_status"][s, :nl], st.ravel()) and np.array_equal(o["lm_next"][s, :nl], p)
            keep = st.ravel() == 1
        else:
            keep = np.zeros(0, bool)
        if keep.sum() < 4:
            assert o["pnp_ok"][s] == 0 and o["n_inliers"][s] == 0 and not o["inlier_mask"][s].any()
        else:
            ok, rv, tv, inl = cv2_compat.solvePnPRansac(wl.lm_obj[0, s, :nl][keep], p[keep], wl.K, np.zeros(4),
                                                        flags=cv2_compat.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                                                        reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
            assert bool(o["pnp_ok"][s]) == ok
            if ok:
                assert int(o["n_inliers"][s]) == len(inl)
                assert np.array_equal(np.flatnonzero(o["inlier_mask"][s]), np.flatnonzero(keep)[inl.ravel()])
    sb.close()


def test_batch_good_features_equals_per_image_call(wl):
    """b200vo_batch_good_features on the resident frames == cv2.goodFeaturesToTrack per image (reference :256 options)."""
    opts = workload.REFERENCE_OPTIONS["kitti"]
    sb = SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                       max_landmarks=wl.L, max_candidates=wl.Cn)
    sb.prime(wl.frames[0])
    for frame_idx, (mc, q, md) in ((0, (1400, 0.1, 10.0)), (1, (300, 0.03, 7.0))):
        if frame_idx:     # after a step the NEW frames are the resident ones
            sb.step(wl.frames[1], wl.lm_pts[0], wl.lm_obj[0], wl.n_lm[0], wl.cand_pts[0], wl.n_cand[0])
        corners, n = sb.good_features(mc, q, md)
        assert corners.shape == (wl.batch, mc, 2) and n.shape == (wl.batch,)
        for s in range(wl.batch):
            ref = cv2_compat.goodFeaturesToTrack(wl.frames[frame_idx, s], mc, q, md, blockSize=3)
            ref = np.zeros((0, 2), np.float32) if ref is None else ref.reshape(-1, 2)
            assert int(n[s]) == len(ref) and np.array_equal(corners[s, :n[s]], ref), (frame_idx, s)
            try:
                import cv2
            except ImportError:
                continue
            c = cv2.goodFeaturesToTrack(wl.frames[frame_idx, s], mc, q, md, blockSize=3)
            assert np.array_equal(corners[s, :n[s]], c.reshape(-1, 2))
    from monocular_visual_odometry_va4mr_b200._lib import B200VOError
    with pytest.raises((B200VOError, NotImplementedError)):
        sb.good_features(0, 0.1, 10.0)
    sb.close()


@pytest.mark.parametrize("batch", [10, 33])
def test_batch_chunked_upload_paths(batch):
    """Batches large enough for the chunked call-by-call upload (ragged last chunk) give the bits of the prefetch form
    and of the per-call path."""
    opts = workload.REFERENCE_OPTIONS["kitti"]
    w2 = workload.TrackWorkload("kitti", batch=batch, n_frames=3, n_landmarks=60, n_candidates=40, n_distinct=2, seed=9,
                                width=320, height=160, cap_landmarks=64, cap_candidates=64)
    order, ref = _run_steps(w2, 3, opts, pinned=True)                 # call by call (chunked)
    sb = SequenceBatch(w2.batch, w2.h, w2.w, w2.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                       pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                       max_landmarks=w2.L, max_candidates=w2.Cn)
    frames = sb.pinned_frames(w2.F)
    frames[:] = w2.frames
    sb.prime(frames[order[0]])
    sb.submit_frames(frames[order[1]])
    for t in range(3):
        f = order[t]
        if t + 2 <= 3:
            sb.submit_frames(frames[order[t + 2]])
        o = sb.step(None, w2.lm_pts[f], w2.lm_obj[f], w2.n_lm[f], w2.cand_pts[f], w2.n_cand[f])
        for s_ in range(batch):                                  # live slots (the others are not written by the kernels)
            nl, nc = int(w2.n_lm[f, s_]), int(w2.n_cand[f, s_])
            for k in ("lm_next", "lm_status", "inlier_mask"):
                assert np.array_equal(o[k][s_, :nl], ref[t][k][s_, :nl]), (t, k, s_)
            for k in ("cand_next", "cand_status"):
                assert np.array_equal(o[k][s_, :nc], ref[t][k][s_, :nc]), (t, k, s_)
        for k in ("pose", "pnp_ok", "n_inliers"):
            assert np.array_equal(o[k], ref[t][k]), (t, k)
    sb.close()
    f, g = order[0], order[1]
    for s in (0, batch // 2, batch - 1):
        nl = int(w2.n_lm[f, s])
        p, st, _ = cv2_compat.calcOpticalFlowPyrLK(w2.frames[f, s], w2.frames[g, s], w2.lm_pts[f, s, :nl], None,
                                                   winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
        assert np.array_equal(ref[0]["lm_status"][s, :nl], st.ravel()) and np.array_equal(ref[0]["lm_next"][s, :nl], p)


# ---- round 2: argument guards, buffer lifetime, and parity at the MEASURED configuration ----
def _mk(wl, opts, **kw):
    return SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                         pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                         max_landmarks=wl.L, max_candidates=wl.Cn, **kw)


def test_counts_beyond_capacity_are_rejected(wl):
    """A count above the slot capacity used to read / write the neighbouring sequence's arrays."""
    import ctypes as C
    from monocular_visual_odometry_va4mr_b200 import _lib
    opts = workload.REFERENCE_OPTIONS["kitti"]
    sb = _mk(wl, opts)
    sb.prime(wl.frames[0])
    bad = wl.n_lm[0].copy()
    bad[1] = wl.L + 5
    with pytest.raises(ValueError):
        sb.step(wl.frames[1], wl.lm_pts[0], wl.lm_obj[0], bad, wl.cand_pts[0], wl.n_cand[0])
    # straight through the C ABI: B200VO_E_BADARG, nothing launched
    p = lambda a, t: a.ctypes.data_as(t)
    for which in ("lm", "cand"):
        n_lm, n_cand = wl.n_lm[0].copy(), wl.n_cand[0].copy()
        if which == "lm":
            n_lm[2] = -1
        else:
            n_cand[0] = wl.Cn + 1
        rc = sb.ctx.lib.b200vo_batch_step(sb.h, p(np.ascontiguousarray(wl.frames[1]), _lib.c_u8p), p(wl.lm_pts[0], _lib.c_f32p),
                                          p(wl.lm_obj[0], _lib.c_f32p), p(n_lm, _lib.c_i32p), p(wl.cand_pts[0], _lib.c_f32p),
                                          p(n_cand, _lib.c_i32p), *sb._out_ptrs)
        assert rc < 0 and "outside" in sb.ctx.last_error()
    # the batch is still usable afterwards
    o = sb.step(wl.frames[1], wl.lm_pts[0], wl.lm_obj[0], wl.n_lm[0], wl.cand_pts[0], wl.n_cand[0])
    assert o["pnp_ok"].all()
    sb.close()


def test_device_counts_are_clamped_to_capacity(wl):
    """The *_dev form cannot validate device-resident counts on the host: the kernels clamp them."""
    import torch
    opts = workload.REFERENCE_OPTIONS["kitti"]
    sb = _mk(wl, opts)
    sb.prime(wl.frames[0])
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    n_bad = wl.n_lm[0].copy()
    n_bad[:] = wl.L + 1000                       # garbage counts
    b, L, Cn = wl.batch, wl.L, wl.Cn
    o = dict(lm_next=torch.zeros((b, L, 2), dtype=torch.float32, device=dev), lm_status=torch.zeros((b, L), dtype=torch.uint8, device=dev),
             cand_next=torch.zeros((b, Cn, 2), dtype=torch.float32, device=dev), cand_status=torch.zeros((b, Cn), dtype=torch.uint8, device=dev),
             pose=torch.zeros((b, 6), dtype=torch.float64, device=dev), pnp_ok=torch.zeros((b,), dtype=torch.uint8, device=dev),
             inlier_mask=torch.zeros((b, L), dtype=torch.uint8, device=dev), n_inliers=torch.zeros((b,), dtype=torch.int32, device=dev))
    guard = torch.full((4096,), 7, dtype=torch.uint8, device=dev)    # allocated right after the outputs
    ins = [t(wl.frames[1]), t(wl.lm_pts[0]), t(wl.lm_obj[0]), t(n_bad), t(wl.cand_pts[0]), t(wl.n_cand[0])]
    sb.step_dev(*[x.data_ptr() for x in ins], {k: v.data_ptr() for k, v in o.items()})
    sb.ctx.sync()
    torch.cuda.synchronize()
    assert int(o["n_inliers"].max()) <= L and bool((guard == 7).all())
    sb.close()


def test_step_dev_refuses_queued_frame_sets(wl):
    import torch
    opts = workload.REFERENCE_OPTIONS["kitti"]
    sb = _mk(wl, opts)
    frames = sb.pinned_frames(wl.F)
    frames[:] = wl.frames
    sb.prime(frames[0])
    sb.submit_frames(frames[1])
    sb.submit_frames(frames[2])
    dev = torch.device("cuda", 0)
    z = torch.zeros(8, dtype=torch.uint8, device=dev).data_ptr()
    with pytest.raises(Exception, match="waiting"):
        sb.step_dev(z, z, z, z, z, z, dict(lm_next=z, lm_status=z, cand_next=z, cand_status=z, pose=z, pnp_ok=z, inlier_mask=z, n_inliers=z))
    # the queued sets are still consumed in order afterwards
    for f in (0, 1):
        sb.step(None, wl.lm_pts[f], wl.lm_obj[f], wl.n_lm[f], wl.cand_pts[f], wl.n_cand[f])
    sb.close()


def test_result_arrays_outlive_the_batch(wl):
    """step() returns views on page-locked memory; they must stay valid after close() / collection of the batch."""
    import gc
    opts = workload.REFERENCE_OPTIONS["kitti"]

    def run():
        sb = _mk(wl, opts)
        sb.prime(wl.frames[0])
        return sb.step(wl.frames[1], wl.lm_pts[0], wl.lm_obj[0], wl.n_lm[0], wl.cand_pts[0], wl.n_cand[0])["pose"]

    pose = run()
    want = pose.copy()
    gc.collect()
    junk = [np.ones(1 << 20, np.uint8) for _ in range(8)]   # churn the allocator
    assert np.array_equal(pose, want) and np.isfinite(pose).all() and len(junk) == 8


def test_profile_rows_on_the_chunked_path(wl):
    """b200vo_batch_profile_read after chunked host steps (batch >= 8) used to time never-recorded events and leave a
    sticky CUDA error behind."""
    from monocular_visual_odometry_va4mr_b200 import _lib
    opts = workload.REFERENCE_OPTIONS["kitti"]
    w8 = workload.TrackWorkload("kitti", batch=8, n_frames=2, n_landmarks=60, n_candidates=40, n_distinct=2, seed=4,
                                width=640, height=240, cap_landmarks=64, cap_candidates=64)
    sb = _mk(w8, opts)
    sb.prime(w8.frames[0])
    sb.ctx.lib.b200vo_batch_profile(sb.h, 1)
    for _ in range(2):
        o = sb.step(w8.frames[1], w8.lm_pts[0], w8.lm_obj[0], w8.n_lm[0], w8.cand_pts[0], w8.n_cand[0])
    ms, n = np.zeros(3, np.float32), np.zeros(1, np.int32)
    assert sb.ctx.lib.b200vo_batch_profile_read(sb.h, ms.ctypes.data_as(_lib.c_f32p), n.ctypes.data_as(_lib.c_intp)) == 0
    assert n[0] == 0 and (ms == 0).all()              # chunked steps have no single pyramid interval: no rows, no error
    sb.ctx.lib.b200vo_batch_profile(sb.h, 0)
    o = sb.step(w8.frames[0], w8.lm_pts[1], w8.lm_obj[1], w8.n_lm[1], w8.cand_pts[1], w8.n_cand[1])   # no spurious failure
    assert o["pnp_ok"].all()
    sb.close()


def test_bench_configuration_parity():
    """The exact workload bench.py times (64 sequences, 1241x376, caps 1024, the reference's KITTI options), 2 steps:
    sequences 0, 21, 42, 63 against the per-call path (bit-equal) and the oracle (bit-equal KLT, identical inlier masks)."""
    import oracle
    import bench
    args = bench.parse([])
    opts = workload.REFERENCE_OPTIONS[args.shape]
    wlb = bench.make_workload(args, 64, 0)
    assert (wlb.batch, wlb.h, wlb.w, wlb.L, wlb.Cn) == (64, 376, 1241, 1024, 1024)
    order, outs = _run_steps(wlb, 2, opts, pinned=True)
    for t, o in enumerate(outs):
        f, g = order[t], order[t + 1]
        for s in (0, 21, 42, 63):
            nl, nc = int(wlb.n_lm[f, s]), int(wlb.n_cand[f, s])
            p, st, _ = cv2_compat.calcOpticalFlowPyrLK(wlb.frames[f, s], wlb.frames[g, s], wlb.lm_pts[f, s, :nl], None,
                                                       winSize=opts["win"], maxLevel=opts["max_level"], criteria=opts["criteria"])
            rp, rst, _ = oracle.calc_optical_flow_pyr_lk(wlb.frames[f, s], wlb.frames[g, s], wlb.lm_pts[f, s, :nl],
                                                         opts["win"], opts["max_level"], opts["criteria"])
            assert np.array_equal(o["lm_status"][s, :nl], st.ravel()) and np.array_equal(st, rst)
            assert np.array_equal(o["lm_next"][s, :nl], p)
            keep = rst.ravel() == 1
            assert np.array_equal(p[keep], rp[keep])
            cp, cst, _ = oracle.calc_optical_flow_pyr_lk(wlb.frames[f, s], wlb.frames[g, s], wlb.cand_pts[f, s, :nc],
                                                         opts["win"], opts["max_level"], opts["criteria"])
            assert np.array_equal(o["cand_status"][s, :nc], cst.ravel())
            ck = cst.ravel() == 1
            assert np.array_equal(o["cand_next"][s, :nc][ck], cp[ck])
            ok, rv, tv, inl, _ = oracle.solve_pnp_ransac_p3p(wlb.lm_obj[f, s, :nl][keep], rp[keep], wlb.K, opts["pnp_iters"],
                                                             opts["pnp_err"], opts["pnp_conf"])
            assert ok and o["pnp_ok"][s]
            assert np.array_equal(np.flatnonzero(o["inlier_mask"][s]), np.flatnonzero(keep)[inl.ravel()])
            assert np.abs(o["pose"][s] - np.concatenate([rv.ravel(), tv.ravel()])).max() <= 1e-6
            ok2, rv2, tv2, inl2 = cv2_compat.solvePnPRansac(wlb.lm_obj[f, s, :nl][keep], p[keep], wlb.K, np.zeros(4),
                                                            flags=cv2_compat.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                                                            reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
            assert np.array_equal(o["pose"][s], np.concatenate([rv2.ravel(), tv2.ravel()]))
