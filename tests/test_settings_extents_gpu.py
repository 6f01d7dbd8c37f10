"""Per-sequence lens distortion and detection masks against the oracle at the frame sizes of test_batch_extents_gpu.py, with
live bytes in the slot padding, on every path that builds a pyramid, and the update rules of the settings (batch.cu's
k_setting) in scripted orders.

Every frame a sequence gets here stands in its slot with random bytes around it, and every slot-layout mask has random
nonzero bytes around the sequence's own mask.  remap is BORDER_CONSTANT 0, so a map tap outside a sequence's frame reads 0
and a mask byte outside it is never read: a gather, a detector maximum or a staging copy bounded by the slot instead of the
sequence's size reads those bytes and changes the result.  Outward models (plumb, pincushion, rational) map part of an
undistorted frame outside the raw one, which is where the padding lies.  A distorted sequence is compared with the oracle on
its cv2.undistort-ed tight frame (tests/undistort_reference.py) and a masked one with tests/mask_reference.py."""
import numpy as np
import pytest

import mask_reference as R
import oracle
import undistort_reference as U
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT
from monocular_visual_odometry_va4mr_b200 import synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch, initial_state, match_bootstrap_frames
from test_batch_extents_gpu import (GFTT_CASES, SIZE_TABLE, SLOT, VO_BORDER, _corner_images, _crops, _levels, _percall_step,
                                    _slot_layout, _track_points, sizes_for)

CHUNKS = 4                                   # batch.cuh B200VO_BATCH_CHUNKS: a host step of 2 * CHUNKS or more sequences
MODEL_CYCLE = list(U.MODELS) + [None]        # goes up in CHUNKS chunks of ceil(batch / CHUNKS) sequences
OUTWARD = ("plumb_4", "pincushion_5", "rational_8", "rational_pole_8")   # models that map part of the frame outside it
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
TRACK_KEYS = ("lm_next", "lm_status", "cand_next", "cand_status")
STEP_KEYS = TRACK_KEYS + ("pose", "pnp_ok", "inlier_mask", "n_inliers")


def _K_for(size, k):
    """the KITTI camera scaled to the size, with a fractional principal point that depends on k"""
    r, c = size
    return U.scale_K(synth.K_KITTI, r, c, 376, 1241, ((k % 4) * 0.25 - 0.375, (k % 3) * 0.3125 - 0.3))


def _d8(model):
    return U.dist8(None if model is None else U.MODELS[model])


def _distorted(model):
    return model is not None and any(U.MODELS[model])


def _und(img, K, model):
    return img if model is None else U.undistort(img, K, U.MODELS[model])


def _outside_taps(K, model, size, slot=SLOT):
    """the map taps of nonzero weight that fall outside the frame but inside its slot"""
    r, c = size
    xy, fr = U.undistort_map(K, U.MODELS[model], r, c)
    x, y, fr = xy[..., 0].astype(np.int64), xy[..., 1].astype(np.int64), fr.astype(np.int64)
    ax, ay = fr & 31, fr >> 5
    n = 0
    for dx, dy, wgt in ((0, 0, (32 - ax) * (32 - ay)), (1, 0, ax * (32 - ay)), (0, 1, (32 - ax) * ay), (1, 1, ax * ay)):
        tx, ty = x + dx, y + dy
        n += int(((wgt > 0) & (tx >= 0) & (ty >= 0) & (tx < slot[1]) & (ty < slot[0]) & ((tx >= c) | (ty >= r))).sum())
    return n


def _mask_layout(masks, rng, slot):
    """per-sequence masks as the top-left of slot-sized masks whose other bytes are random and nonzero"""
    out = rng.integers(1, 256, (len(masks),) + tuple(slot), dtype=np.uint8)
    for k, m in enumerate(masks):
        out[k, :m.shape[0], :m.shape[1]] = m
    return out


def _copy(r):
    return {k: np.array(v) for k, v in r.items()}


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def _same(ra, rb, keys):
    for k in keys:
        assert np.array_equal(ra[k], rb[k], equal_nan=True), k


# ---------------------------------------------------------------------------------------------------- the cases
# the tracker: the two staged kernels and one generic one
TRACK_CASES = [((15, 15), 5, (3, 50, 0.01)), ((21, 21), 3, (3, 30, 0.01)), ((9, 13), 4, (3, 20, 0.001))]


def _track_models(sizes):
    return [MODEL_CYCLE[k % len(MODEL_CYCLE)] for k in range(len(sizes))]


# the chunked host step: 13 sequences go up in chunks of 4, 4, 4 and 1; distortion only in the second and the last
CHUNK_SIZES = [(376, 1241), (370, 1226), (240, 321), (97, 161), (376, 1242), (353, 1025), (61, 129), (33, 383),
               (375, 1242), (257, 513), (120, 640), (17, 129), (240, 320)]
CHUNK_MODELS = {4: "plumb_4", 5: "pincushion_5", 6: "rational_pole_8", 12: "kitti_like_5"}


def _chunk_of(b, n):
    per = -(-n // CHUNKS)
    return b // per


# the detector: mask kinds cycled over the sequences, every third sequence distorted
MASK_KINDS = ["hood", "blob", "corner_pixels", "ring", "zero", "padding_only", "fused_split", None]
GFTT_MODELS = ["pincushion_5", "plumb_4", "rational_8", "kitti_like_5"]


def _gftt_layout(sizes):
    kinds = [MASK_KINDS[k % len(MASK_KINDS)] for k in range(len(sizes))]
    models = [GFTT_MODELS[(k // 3) % len(GFTT_MODELS)] if k % 3 == 1 else None for k in range(len(sizes))]
    return kinds, models


def _tight_mask(kind, img, k):
    """the in-frame part of a mask of the given kind for the (undistorted) image"""
    r, c = img.shape
    if kind == "hood":
        return R.hood_mask((r, c))
    if kind == "blob":
        return R.blob_mask((r, c), seed=k)
    m = np.zeros((r, c), np.uint8)
    if kind == "corner_pixels":
        # the three weakest candidates at a low quality: their masked maximum lies far under the image's own
        idx, w = R.gftt_candidates(img, 0.001)
        for a in idx[-3:].tolist():
            m[a // w, a % w] = 255
        m[r // 2, c // 2] = 255
    elif kind == "ring":
        m[0, :] = m[-1, :] = m[:, 0] = m[:, -1] = 255
    elif kind == "fused_split":
        x = c & ~31
        m[:, max(x - 3, 0):x + 3] = 200
    return m                    # "zero" and "padding_only": nothing inside the frame


# the bootstrap: the interleaved layout of test_bootstrap_interleaved_sizes with two widths that are not multiples of 4
A, B, C, D, E = (376, 1241), (370, 1226), (240, 321), (33, 31), (97, 161)
BOOT_LAYOUT = [A, B, C, A, D, A, B, A, E, A, B, A, A, C, A, A, A, A, A, A, A]
BOOT_MODELS = {0: "kitti_like_5", 2: "plumb_4", 5: "plumb_4", 8: "plumb_4", 13: "kitti_like_5", 17: "plumb_4", 19: "kitti_like_5"}
BOOT_MASKS = {1: "hood", 5: "blob", 8: "hood", 13: "blob", 18: "hood", 19: "blob"}
BOOT_LISTED = [11, 2, 4, 0, 8, 6, 19, 13, 17]


def _boot_K(size):
    return {A: synth.K_KITTI, B: np.array([[707.0912, 0, 601.8873], [0, 707.0912, 183.1104], [0, 0, 1.0]]),
            C: np.array([[300.0, 0, 160.25], [0, 300.0, 123.25], [0, 0, 1.0]]), D: np.array([[40.0, 0, 15.0], [0, 40.0, 19.75], [0, 0, 1.0]]),
            E: np.array([[120.0, 0, 80.25], [0, 120.0, 51.5], [0, 0, 1.0]])}[size]


# ---------------------------------------------------------------------------------------------------- the table itself (CPU)
def test_settings_table_covers_its_edges():
    """What the cases below rest on, checked with the oracle's map and plain arithmetic."""
    for win, ml, crit in TRACK_CASES:
        sizes = sizes_for(win)
        models = _track_models(sizes)
        assert set(U.MODELS) <= set(models) and None in models, win
        assert {"rational_pole_8", "zero_5"} <= set(models)
        n_out = 0
        for k, (size, m) in enumerate(zip(sizes, models)):
            if m is None:
                continue
            taps = _outside_taps(_K_for(size, k), m, size)
            if m in OUTWARD and size != SLOT:
                assert taps > 0, (win, size, m)       # live padding under the gather
                n_out += 1
        assert n_out >= 6, win
        # a distorted sequence under VO_BORDER + 2 rows, with taps in its padding: REFLECT_101 bounces more than once
        assert any(m in OUTWARD and r < VO_BORDER + 2 and _outside_taps(_K_for((r, c), k), m, (r, c)) > 0
                   for k, ((r, c), m) in enumerate(zip(sizes, models))), win
        # one-level pyramids and widths where the pad kernel's 16-byte stores straddle w + VO_BORDER
        assert any(_distorted(m) and _levels(s, win, ml) == 1 for s, m in zip(sizes, models)), win
        assert any(_distorted(m) and (s[1] + VO_BORDER) % 16 for s, m in zip(sizes, models)), win
    # the chunked step: distortion in a chunk other than the first, and in the last chunk, which holds one sequence
    n = len(CHUNK_SIZES)
    assert n >= 3 * CHUNKS and len(set(CHUNK_SIZES)) == n
    chunks = {_chunk_of(b, n) for b in CHUNK_MODELS}
    assert 0 not in chunks and chunks == {1, _chunk_of(n - 1, n)} and _chunk_of(n - 1, n) == CHUNKS - 1
    assert sum(_chunk_of(b, n) == CHUNKS - 1 for b in range(n)) == 1
    assert any(_outside_taps(_K_for(CHUNK_SIZES[b], b), m, CHUNK_SIZES[b]) > 0 for b, m in CHUNK_MODELS.items())
    # every mask kind, distorted sequences among the masked ones, the padding always live
    for max_corners, quality, min_dist, slot in GFTT_CASES:
        sizes = [s for s in sizes_for((5, 7)) if s[0] <= slot[0] and s[1] <= slot[1]]
        sizes += [slot] * (slot not in sizes)
        kinds, models = _gftt_layout(sizes)
        assert set(MASK_KINDS) <= set(kinds) or len(sizes) < len(MASK_KINDS)
        assert any(m is not None and kd is not None for kd, m in zip(kinds, models))
        assert any(m in OUTWARD and s != slot and _outside_taps(_K_for(s, k), m, s, slot) > 0
                   for k, (s, m) in enumerate(zip(sizes, models)))
        rng = np.random.default_rng(0)
        tight = [_tight_mask(kd or "zero", np.full(s, 9, np.uint8), k) for k, (s, kd) in enumerate(zip(sizes, kinds))]
        lay = _mask_layout(tight, rng, slot)
        for k, (r, c) in enumerate(sizes):
            pad = np.concatenate([lay[k, r:, :].ravel(), lay[k, :r, c:].ravel()])
            assert (r, c) == slot or (pad.size and pad.all()), (slot, (r, c))
    # the bootstrap: distortion and masks in both SIFT chunks of the KITTI 00-02 group, widths not multiples of 4
    a_seqs = [s for s, size in enumerate(BOOT_LAYOUT) if size == A]
    assert len(a_seqs) >= 14
    for part in (a_seqs[:len(a_seqs) // 2], a_seqs[len(a_seqs) // 2:]):
        assert set(part) & set(BOOT_MODELS) and set(part) & set(BOOT_MASKS)
    assert {C[1] % 4, E[1] % 4} == {1}
    assert {BOOT_LAYOUT[s] for s in BOOT_MODELS} >= {A, C, E} and BOOT_LISTED != sorted(BOOT_LISTED)
    assert set(BOOT_LISTED) & set(BOOT_MODELS) and set(BOOT_LISTED) & set(BOOT_MASKS)
    for s, m in BOOT_MODELS.items():
        if m in OUTWARD:
            assert _outside_taps(_boot_K(BOOT_LAYOUT[s]), m, BOOT_LAYOUT[s]) > 0, s
    assert all(size in SIZE_TABLE for size in (A, B, D))


# ---------------------------------------------------------------------------------------------------- shared inputs
@pytest.fixture(scope="module")
def slot_frames():
    """Three consecutive KITTI frames at the slot size; a sequence's raw image is a crop of them."""
    return synth.render_sequence("kitti", 3, seed=911, width=SLOT[1], height=SLOT[0])["frames"]


def _points(sizes, win, max_level, rng):
    """landmark and candidate points of every sequence (the edge points of _track_points), packed"""
    n_lv = [_levels(s, win, max_level) for s in sizes]
    lm = [_track_points(s, win, n, rng) for s, n in zip(sizes, n_lv)]
    cand = [_track_points(s, win, n, rng)[::-1].copy() for s, n in zip(sizes, n_lv)]
    L, Cn, b = max(len(p) for p in lm), max(len(p) for p in cand), len(sizes)
    lm_pts, cand_pts = np.zeros((b, L, 2), np.float32), np.zeros((b, Cn, 2), np.float32)
    for k in range(b):
        lm_pts[k, :len(lm[k])], cand_pts[k, :len(cand[k])] = lm[k], cand[k]
    lm_obj = np.zeros((b, L, 3), np.float32)
    lm_obj[..., 2] = 10.0
    return lm, cand, (lm_pts, lm_obj, np.int32([len(p) for p in lm]), cand_pts, np.int32([len(p) for p in cand]))


# ---------------------------------------------------------------------------------------------------- tracker
@pytest.mark.gpu
@pytest.mark.parametrize("win,max_level,crit", TRACK_CASES, ids=[f"{w[0]}x{w[1]}" for w, _, _ in TRACK_CASES])
def test_tracker_distorted_against_oracle(slot_frames, win, max_level, crit):
    """Mixed sizes with every distortion model and none: each sequence equals the oracle on its undistorted tight frames,
    and a batch of one at its size, bit for bit."""
    rng = np.random.default_rng(win[0] * 7 + win[1])
    sizes = sizes_for(win)
    models = _track_models(sizes)
    Ks = np.stack([_K_for(s, k) for k, s in enumerate(sizes)])
    raw = _crops(slot_frames, sizes, rng)
    und = [np.stack([_und(f, K, m) for f in fr]) for fr, K, m in zip(raw, Ks, models)]
    lm, cand, args = _points(sizes, win, max_level, rng)
    kw = dict(win=win, max_level=max_level, criteria=crit, max_landmarks=args[0].shape[1], max_candidates=args[3].shape[1])
    mixed = SequenceBatch(len(sizes), *SLOT, Ks, frame_size=sizes, dist_coeffs=[_d8(m) for m in models], **kw)
    assert np.array_equal(mixed.dist_coeffs, [_d8(m) for m in models])
    mixed.prime(_slot_layout([r[0] for r in raw], rng))
    got = [_copy(mixed.step(_slot_layout([r[f] for r in raw], rng), *args)) for f in (1, 2)]
    mixed.close()
    outcomes = set()
    for k, (size, m) in enumerate(zip(sizes, models)):
        one = SequenceBatch(1, *size, Ks[k], dist_coeffs=[_d8(m)], **kw)
        one.prime(raw[k][0][None])
        one_args = [a[k:k + 1].copy() for a in args]
        got_one = [_copy(one.step(raw[k][f][None].copy(), *one_args)) for f in (1, 2)]
        one.close()
        for f in (1, 2):
            for key, pts in (("lm", lm[k]), ("cand", cand[k])):
                n = len(pts)
                rp, rst, _ = oracle.calc_optical_flow_pyr_lk(und[k][f - 1], und[k][f], pts, win, max_level, crit)
                rst = rst.ravel()
                ok = rst == 1
                st, nxt = got[f - 1][f"{key}_status"][k, :n], got[f - 1][f"{key}_next"][k, :n]
                assert np.array_equal(st, rst), (size, m, f, key, np.flatnonzero(st != rst)[:8])
                assert np.array_equal(nxt[ok], rp[ok]), (size, m, f, key)
                assert np.array_equal(st, got_one[f - 1][f"{key}_status"][0, :n]), (size, m, f, key)
                assert np.array_equal(nxt, got_one[f - 1][f"{key}_next"][0, :n]), (size, m, f, key)
                outcomes |= set(rst.tolist())
    assert outcomes == {0, 1}


# ---------------------------------------------------------------------------------------------------- chunked host step
def _chunk_inputs(sizes, rng, n_frames=4):
    Ks = np.stack([_K_for(s, k) for k, s in enumerate(sizes)])
    models = [CHUNK_MODELS.get(k) for k in range(len(sizes))]
    frames = [synth.render_sequence("kitti", n_frames, seed=300 + k, width=c, height=r, K=Ks[k])["frames"]
              for k, (r, c) in enumerate(sizes)]
    und = [[_und(f, K, m) for f in fr] for fr, K, m in zip(frames, Ks, models)]
    return Ks, models, frames, und


@pytest.mark.gpu
@pytest.mark.parametrize("uniform", [False, True], ids=["mixed", "uniform"])
def test_chunked_host_step_distortion_equals_undistorted_input(uniform):
    """13 sequences, distortion only in the second chunk and in the last one: host steps (chunked), submitted sets and
    step_dev equal, bit for bit, the same batch fed the undistorted frames.  uniform: every sequence at the slot size, so
    the batch has no extent table."""
    import torch
    rng = np.random.default_rng(13 + uniform)
    sizes = [SLOT] * len(CHUNK_SIZES) if uniform else CHUNK_SIZES
    n = len(sizes)
    Ks, models, raw, und = _chunk_inputs(sizes, rng)
    _, _, args = _points(sizes, (15, 15), 5, rng)
    kw = dict(max_landmarks=args[0].shape[1], max_candidates=args[3].shape[1])
    a = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, dist_coeffs=[_d8(m) for m in models], **kw)
    b = SequenceBatch(n, *SLOT, Ks, frame_size=sizes, **kw)

    def pair(f):
        pad = rng.integers(0, 256, (n,) + SLOT, dtype=np.uint8)
        fa, fb = pad.copy(), pad.copy()
        for k, (r, c) in enumerate(sizes):
            fa[k, :r, :c], fb[k, :r, :c] = raw[k][f], und[k][f]
        return fa, fb

    def same_features():
        ca, na = a.good_features(1400, 0.1, 10.0)
        cb, nb = b.good_features(1400, 0.1, 10.0)
        assert np.array_equal(na, nb) and np.array_equal(ca, cb)
        return na

    fa, fb = pair(0)
    a.prime(fa)
    b.prime(fb)
    assert same_features()[list(CHUNK_MODELS)].all()
    # host step: the frames go up in CHUNKS chunks
    fa, fb = pair(1)
    _same(_copy(a.step(fa, *args)), b.step(fb, *args), STEP_KEYS)
    same_features()
    # submitted sets, consumed by step(None)
    fa, fb = pair(2)
    pa, pb = a.pinned_frames()[0], b.pinned_frames()[0]
    pa[...], pb[...] = fa, fb
    a.submit_frames(pa)
    b.submit_frames(pb)
    _same(_copy(a.step(None, *args)), b.step(None, *args), STEP_KEYS)
    same_features()
    # step_dev on device frames
    fa, fb = pair(3)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    ins = [dev(x) for x in args]
    outs = []
    for sb, f in ((a, fa), (b, fb)):
        o = {k: torch.zeros(v.shape, dtype=getattr(torch, str(v.dtype)), device="cuda") for k, v in sb._out_dict.items()}
        fd = dev(f)
        torch.cuda.synchronize()
        sb.step_dev(fd.data_ptr(), *(x.data_ptr() for x in ins), {k: v.data_ptr() for k, v in o.items()})
        sb.ctx.sync()
        outs.append({k: v.cpu().numpy() for k, v in o.items()})
    _same(outs[0], outs[1], STEP_KEYS)
    same_features()
    a.close()
    b.close()


# ---------------------------------------------------------------------------------------------------- detector
@pytest.mark.gpu
@pytest.mark.parametrize("max_corners,quality,min_dist,slot", GFTT_CASES)
def test_detector_masked_and_distorted_against_oracle(slot_frames, max_corners, quality, min_dist, slot):
    """Every mask kind, some sequences distorted, padding of frames and masks random: each sequence equals
    mask_reference.good_features_to_track on its undistorted tight image with its tight mask."""
    rng = np.random.default_rng(int(min_dist * 1000 + max_corners) + 1)
    sizes = [s for s in sizes_for((5, 7)) if s[0] <= slot[0] and s[1] <= slot[1]]
    sizes += [slot] * (slot not in sizes)
    kinds, models = _gftt_layout(sizes)
    Ks = np.stack([_K_for(s, k) for k, s in enumerate(sizes)])
    raw = _corner_images([c[0] for c in _crops(slot_frames, sizes, rng)], rng)
    und = [_und(im, K, m) for im, K, m in zip(raw, Ks, models)]
    tight = [None if kd is None else _tight_mask(kd, im, k) for k, (kd, im) in enumerate(zip(kinds, und))]
    sb = SequenceBatch(len(sizes), *slot, Ks, win=(5, 7), max_landmarks=4, max_candidates=0, frame_size=sizes,
                       dist_coeffs=[_d8(m) for m in models])
    masked = [k for k, m in enumerate(tight) if m is not None]
    sb.set_detection_mask(masked, _mask_layout([tight[k] for k in masked], rng, slot))
    assert list(np.flatnonzero(sb.has_mask)) == masked
    sb.prime(_slot_layout(raw, rng, slot))
    corners, n = sb.good_features(max_corners, quality, min_dist)
    sb.close()
    for k, (size, im) in enumerate(zip(sizes, und)):
        want = R.good_features_to_track(im, max_corners, quality, min_dist, mask=tight[k])
        want = np.zeros((0, 2), np.float32) if want is None else want.reshape(-1, 2)
        assert n[k] == len(want), (size, kinds[k], models[k], n[k], len(want))
        assert np.array_equal(corners[k, :n[k]], want), (size, kinds[k], models[k])
        if kinds[k] in ("zero", "padding_only", "ring"):
            assert n[k] == 0, (size, kinds[k])
    assert n.sum() > 0
    assert any(n[k] for k in range(len(sizes)) if models[k] is not None and kinds[k] is not None)


# ---------------------------------------------------------------------------------------------------- bootstrap
def _host_chain(K, f0, f1, mask):
    """the host bootstrap chain on undistorted frames with the mask; None where it raises"""
    try:
        return initial_state(K, OPT, *match_bootstrap_frames(f0, f1, OPT["feature_ratio"], mask=mask))
    except Exception:
        return None


@pytest.mark.gpu
def test_bootstrap_distorted_and_masked_interleaved_sizes():
    rng = np.random.default_rng(97)
    n = len(BOOT_LAYOUT)
    Ks = np.stack([_boot_K(s) for s in BOOT_LAYOUT])
    models = [BOOT_MODELS.get(s) for s in range(n)]
    raw = [synth.render_sequence("kitti", 5, seed=520 + s, width=c, height=r, K=Ks[s])["frames"] for s, (r, c) in enumerate(BOOT_LAYOUT)]
    und = [[_und(f, Ks[s], models[s]) for f in fr] for s, fr in enumerate(raw)]
    masks = [None] * n
    for s, kind in BOOT_MASKS.items():
        masks[s] = _tight_mask(kind, und[s][0], s)
    masked = sorted(BOOT_MASKS)
    dev = VOBatch(n, *SLOT, Ks, OPT, frame_size=BOOT_LAYOUT, dist_coeffs=[_d8(m) for m in models], **CAPS)
    host = VOBatch(n, *SLOT, Ks, OPT, frame_size=BOOT_LAYOUT, **CAPS)     # the twin: undistorted frames, host states
    for vb in (dev, host):
        vb.set_detection_mask(masked, _mask_layout([masks[s] for s in masked], rng, SLOT))
    r = _copy(dev.bootstrap(_slot_layout([fr[0] for fr in raw], rng), _slot_layout([fr[2] for fr in raw], rng)))
    ok = []
    for s in range(n):
        st = _host_chain(Ks[s], und[s][0], und[s][2], masks[s])
        if st is None:
            assert r["status"][s] == VOBatch.NO_BOOTSTRAP and r["num_pts"][s] == 0, s
            continue
        assert r["status"][s] == VOBatch.OK and r["num_pts"][s] == st["num_pts"], s
        assert r["n_lm"][s] == len(st["lm"]) and r["n_cand"][s] == len(st["keys"]), s
        _assert_state(dev.read_state(s), st)
        host.load(s, und[s][2], st)
        ok.append(s)
    assert r["status"][BOOT_LAYOUT.index(D)] == VOBatch.NO_BOOTSTRAP
    assert {s for s in BOOT_MODELS if BOOT_LAYOUT[s] != E} <= set(ok) and len(ok) >= n - 3
    # the resident frame is the undistorted second bootstrap frame
    rd = _copy(dev.step(_slot_layout([fr[3] for fr in raw], rng)))
    rh = _copy(host.step(_slot_layout([fr[3] for fr in und], rng)))
    for k in rd:
        assert np.array_equal(rd[k][ok], rh[k][ok]), k

    # a subset in non-monotone order, on frames 1 and 4: again the host chain
    r = _copy(dev.bootstrap(_slot_layout([raw[s][1] for s in BOOT_LISTED], rng), _slot_layout([raw[s][4] for s in BOOT_LISTED], rng),
                            seqs=BOOT_LISTED))
    for k, s in enumerate(BOOT_LISTED):
        st = _host_chain(Ks[s], und[s][1], und[s][4], masks[s])
        if st is None:
            assert r["status"][k] == VOBatch.NO_BOOTSTRAP and dev.read_state(s)["status"] == VOBatch.NO_BOOTSTRAP, s
            continue
        assert r["status"][k] == VOBatch.OK and r["num_pts"][k] == st["num_pts"], s
        assert r["n_lm"][k] == len(st["lm"]) and r["n_cand"][k] == len(st["keys"]), s
        _assert_state(dev.read_state(s), st)
    assert (r["status"] == VOBatch.OK).sum() >= len(BOOT_LISTED) - 2
    for s in set(range(n)) - set(BOOT_LISTED):      # untouched: as the twin that never got the call
        a, b = dev.read_state(s), host.read_state(s)
        _assert_state(a, b)
        assert a["status"] == (b["status"] if s in ok else VOBatch.NO_BOOTSTRAP), s
    dev.close()
    host.close()


# ---------------------------------------------------------------------------------------------------- VOBatch.load at seq > 0
@pytest.mark.gpu
def test_load_distorted_sequence_after_the_first():
    """load(seq > 0) of distorted sequences in a mixed batch, then steps: each sequence equals the per-call path on its
    undistorted frames."""
    rng = np.random.default_rng(5)
    sizes = [(376, 1241), (370, 1226), (240, 321), (376, 1241)]
    models = [None, "plumb_4", "kitti_like_5", "pincushion_5"]
    Ks = np.stack([synth.K_KITTI if s == (376, 1241) else _K_for(s, k) for k, s in enumerate(sizes)])
    n_frames = 9
    raw = [synth.render_sequence("kitti", n_frames, seed=610 + k, width=c, height=r, K=Ks[k])["frames"] for k, (r, c) in enumerate(sizes)]
    und = [[_und(f, Ks[k], models[k]) for f in fr] for k, fr in enumerate(raw)]
    vb = VOBatch(len(sizes), *SLOT, Ks, OPT, frame_size=sizes, dist_coeffs=[_d8(m) for m in models], **CAPS)
    # a step with nothing loaded leaves random bytes around every frame of the device's staging
    r = vb.step(_slot_layout([fr[0] for fr in raw], rng))
    assert (r["status"] == VOBatch.IDLE).all()
    ref = []
    for s in range(len(sizes)):
        st = initial_state(Ks[s], OPT, *match_bootstrap_frames(und[s][0], und[s][2], OPT["feature_ratio"]))
        ref.append({k: st[k] for k in STATE_KEYS})
    for s in (2, 3, 1, 0):
        vb.load(s, raw[s][2], ref[s])
    live = [True] * len(sizes)
    for f in range(3, n_frames):
        r = _copy(vb.step(_slot_layout([fr[f] for fr in raw], rng)))
        for s in range(len(sizes)):
            if not live[s]:
                assert r["status"][s] != VOBatch.OK
                continue
            code, n_inl, host, new = _percall_step(ref[s], und[s][f - 1], und[s][f], Ks[s], r["pose_cw"][s].copy(), OPT)
            assert r["status"][s] == code and r["n_inliers"][s] == n_inl, (s, f)
            if code != VOBatch.OK:
                live[s] = False
                continue
            assert np.abs(r["pose_cw"][s] - host).max() <= 1e-12, (s, f)
            _assert_state(vb.read_state(s), new)
            ref[s] = new
    vb.close()
    assert sum(live[1:]) >= 2, "too few distorted sequences ran every step for the comparison to mean much"


# ---------------------------------------------------------------------------------------------------- settings orders
SSLOT = (240, 400)
SIZES0 = [(240, 400), (200, 321), (97, 161), (240, 400), (161, 257), (120, 399)]
MODELS0 = {1: "plumb_4", 2: "pincushion_5", 4: "kitti_like_5"}
MASKS0 = {0: "hood", 2: "blob", 5: "blob"}
# scripts of setter calls from the settings above: (setter, listed sequences, one value per listed sequence or None);
# K values are indices into _script_K, mask values kinds of _tight_mask, distortion values model names or "zeros"
SCRIPTS = {
    "shrink_grow_shrink": [("size", [2], [(33, 31)]), ("mask", [2], ["hood"]), ("size", [2], [(240, 400)]), ("mask", [2], ["blob"]),
                           ("size", [2], [(61, 129)]), ("mask", [2], ["corner_pixels"])],
    "K_of_distorted": [("K", [1, 3], [1, 2]), ("K", [2], [3])],
    "clear_by_none_and_zero_row": [("dist", [1], None), ("dist", [2], ["zeros"])],
    "last_ones_dropped_and_back": [("mask", [5, 0, 2], None), ("dist", [4, 1, 2], None), ("dist", [3], ["rational_pole_8"]),
                                   ("mask", [4], ["ring"]), ("mask", [1, 4], ["hood", "blob"])],
    "non_monotone_subsets": [("size", [4, 1, 3], [(33, 383), (97, 161), (17, 129)]), ("dist", [5, 0, 3], ["pincushion_5", "plumb_4", "rational_8"]),
                             ("mask", [3, 0, 5], ["blob", "hood", "fused_split"]), ("K", [5, 2, 0], [1, 2, 3]),
                             ("size", [0, 5], [(200, 321), (45, 33)]), ("mask", [5, 0], ["hood", "blob"])],
    "refused_while_waiting": [("wait", None, None)],
}


def _script_K(i, size):
    return _K_for(size, 0) if i == 0 else _K_for(size, i) + np.array([[0, 0, 1.5 * i], [0, 0, -0.75 * i], [0, 0, 0]])


class _Model:
    """the settings a batch should hold, in plain Python"""

    def __init__(self):
        n = len(SIZES0)
        self.size = list(SIZES0)
        self.K = [_script_K(0, SIZES0[s]) for s in range(n)]
        self.dist = [_d8(MODELS0.get(s)) for s in range(n)]
        self.mask = [None if s not in MASKS0 else (MASKS0[s], SIZES0[s]) for s in range(n)]


def _apply(bat, model, op, seqs, vals, frames0, rng):
    """one setter call on the batch and the model"""
    if op == "size":
        bat.set_frame_size(seqs, vals)
        for s, v in zip(seqs, vals):
            model.size[s], model.mask[s] = tuple(v), None
    elif op == "K":
        Ks = np.stack([_script_K(v, model.size[s]) for s, v in zip(seqs, vals)])
        bat.set_intrinsics(seqs, Ks)
        for s, K in zip(seqs, Ks):
            model.K[s] = K
    elif op == "dist":
        if vals is None:
            bat.set_distortion(seqs, None)
        else:
            rows = [np.zeros(4) if v == "zeros" else np.asarray(U.MODELS[v]) for v in vals]
            if len({len(r) for r in rows}) > 1:        # rows of one call have one length
                rows = [U.dist8(r) for r in rows]
            bat.set_distortion(seqs, rows)
        for k, s in enumerate(seqs):
            model.dist[s] = _d8(None if vals is None or vals[k] == "zeros" else vals[k])
    elif op == "mask":
        if vals is None:
            bat.set_detection_mask(seqs, None)
        else:
            tight = [_tight_mask(v, frames0[s][:model.size[s][0], :model.size[s][1]], s) for s, v in zip(seqs, vals)]
            bat.set_detection_mask(seqs, _mask_layout(tight, rng, SSLOT))
        for k, s in enumerate(seqs):
            model.mask[s] = None if vals is None else (vals[k], model.size[s])


def _mirrors_match(bat, model):
    assert np.array_equal(bat.frame_size, model.size)
    assert list(bat.has_mask) == [m is not None for m in model.mask]
    assert np.array_equal(bat.dist_coeffs, model.dist)


def _refusals_while_waiting(bat, model, frames0, rng):
    """with a submitted set waiting: K is refused when a listed sequence is distorted, frame size and distortion always,
    masks never; a refused call changes nothing"""
    dist = [s for s in range(len(SIZES0)) if model.dist[s].any()]
    plain = [s for s in range(len(SIZES0)) if not model.dist[s].any()]
    assert dist and plain
    for op, seqs, vals in (("K", [plain[0], dist[0]], [2, 2]), ("K", dist[:1], [3]), ("size", plain[:1], [(97, 161)]),
                           ("size", dist[:1], [model.size[dist[0]]]), ("dist", plain[:1], ["plumb_4"]), ("dist", dist[:1], None),
                           ("dist", [plain[-1], dist[-1]], ["zeros", "zeros"])):
        before = (bat.frame_size.copy(), bat.has_mask.copy(), bat.dist_coeffs.copy())
        with pytest.raises(ValueError, match="submitted frame sets are waiting"):
            _apply(bat, _Model(), op, seqs, vals, frames0, rng)
        assert all(np.array_equal(x, y) for x, y in zip(before, (bat.frame_size, bat.has_mask, bat.dist_coeffs))), (op, seqs)
    # accepted: K of sequences without distortion, and masks
    _apply(bat, model, "K", plain[::-1], [1] * len(plain), frames0, rng)
    _apply(bat, model, "mask", [dist[-1], plain[0]], ["hood", "fused_split"], frames0, rng)
    _apply(bat, model, "mask", [2], None, frames0, rng)
    _mirrors_match(bat, model)


def _script_frames(rng, n_frames):
    """per sequence: n_frames KITTI frames at the slot size (a sequence's image is their top-left at its size)"""
    K = _script_K(0, SSLOT)
    return [synth.render_sequence("kitti", n_frames, seed=800 + s, width=SSLOT[1], height=SSLOT[0], K=K)["frames"]
            for s in range(len(SIZES0))]


def _layout(frames, model, f, rng):
    out = rng.integers(0, 256, (len(frames),) + SSLOT, dtype=np.uint8)
    for s, (r, c) in enumerate(model.size):
        out[s, :r, :c] = frames[s][f][:r, :c]
    return out


def _fresh(cls, model, frames0, rng):
    """a batch built with the model's settings from the start"""
    kw = dict(win=(15, 15), max_level=3, max_landmarks=512, max_candidates=512) if cls is SequenceBatch else dict(CAPS)
    args = (OPT,) if cls is VOBatch else ()
    bat = cls(len(SIZES0), *SSLOT, np.stack(model.K), *args, frame_size=model.size, dist_coeffs=model.dist, **kw)
    masked = [s for s, m in enumerate(model.mask) if m is not None]
    if masked:
        tight = [_tight_mask(model.mask[s][0], frames0[s][:model.size[s][0], :model.size[s][1]], s) for s in masked]
        bat.set_detection_mask(masked, _mask_layout(tight, rng, SSLOT))
    return bat


def _outcome(bat, model, frames, rng_seed):
    """prime / bootstrap, one step and the detector's corners, each with the same random padding for both batches"""
    rng = np.random.default_rng(rng_seed)
    if isinstance(bat, SequenceBatch):
        sizes = model.size
        _, _, args = _points(sizes, (15, 15), 3, rng)
        L, Cn, b = bat.L, bat.Cn, len(sizes)
        pad = [np.zeros((b, L, 2), np.float32), np.zeros((b, L, 3), np.float32), args[2], np.zeros((b, Cn, 2), np.float32), args[4]]
        pad[0][:, :args[0].shape[1]], pad[1][:, :args[1].shape[1]], pad[3][:, :args[3].shape[1]] = args[0], args[1], args[3]
        bat.prime(_layout(frames, model, 0, rng))
        out = _copy(bat.step(_layout(frames, model, 1, rng), *pad))
        c, n = bat.good_features(300, 0.05, 7.0)
        out.update(corners=c, n_corners=n)
        return out
    out = {f"boot_{k}": v for k, v in _copy(bat.bootstrap(_layout(frames, model, 0, rng), _layout(frames, model, 2, rng))).items()}
    out.update({f"step_{k}": v for k, v in _copy(bat.step(_layout(frames, model, 3, rng))).items()})
    for s in range(bat.batch):
        st = bat.read_state(s)
        out.update({f"{s}_{k}": np.asarray(v) for k, v in st.items()})
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("cls", [SequenceBatch, VOBatch], ids=["SequenceBatch", "VOBatch"])
@pytest.mark.parametrize("script", list(SCRIPTS))
def test_settings_orders(cls, script):
    """A script of setter calls: the mirrors equal a plain model, unlisted sequences keep their settings, refusals while a
    submitted set waits follow k_setting, and the batch computes, bit for bit, what a batch built with the final settings
    computes."""
    rng = np.random.default_rng(len(script))
    frames = _script_frames(rng, 4)
    frames0 = [fr[0] for fr in frames]
    model = _Model()
    bat = _fresh(cls, model, frames0, rng)
    _mirrors_match(bat, model)
    for op, seqs, vals in SCRIPTS[script]:
        before = _Model()
        before.__dict__ = {k: list(v) for k, v in model.__dict__.items()}
        if op == "wait":
            # a submitted set waits: the refusals, then the set is consumed
            if cls is SequenceBatch:
                bat.prime(_layout(frames, model, 0, rng))
                p = bat.pinned_frames()[0]
                p[...] = _layout(frames, model, 1, rng)
                bat.submit_frames(p)
                _refusals_while_waiting(bat, model, frames0, rng)
                z = np.zeros((bat.batch, bat.L, 2), np.float32)
                bat.step(None, z, np.zeros((bat.batch, bat.L, 3), np.float32), np.zeros(bat.batch, np.int32),
                         np.zeros((bat.batch, bat.Cn, 2), np.float32), np.zeros(bat.batch, np.int32))
            else:
                p = bat.pinned_frames()[0]
                p[...] = _layout(frames, model, 1, rng)
                bat.submit_frames(p)
                _refusals_while_waiting(bat, model, frames0, rng)
                bat.step(None)
            continue
        _apply(bat, model, op, seqs, vals, frames0, rng)
        _mirrors_match(bat, model)
        for s in set(range(len(SIZES0))) - set(seqs):          # unlisted sequences keep every setting
            assert model.size[s] == before.size[s] and np.array_equal(model.dist[s], before.dist[s])
            assert np.array_equal(model.K[s], before.K[s]) and model.mask[s] == before.mask[s]
            assert tuple(bat.frame_size[s]) == tuple(before.size[s]) and np.array_equal(bat.dist_coeffs[s], before.dist[s])
            assert bat.has_mask[s] == (before.mask[s] is not None)
    fresh = _fresh(cls, model, frames0, np.random.default_rng(len(script)))
    # the masks of both batches hold the same in-frame bytes (the padding differs and is never read)
    got, want = _outcome(bat, model, frames, 42), _outcome(fresh, model, frames, 42)
    assert got.keys() == want.keys()
    for k in got:
        assert np.array_equal(got[k], want[k], equal_nan=True), k
    bat.close()
    fresh.close()


@pytest.mark.gpu
def test_set_intrinsics_of_a_running_distorted_sequence_keeps_its_pyramid():
    """Today's behaviour: set_intrinsics on a running distorted VOBatch sequence keeps its resident pyramid (undistorted
    with the old K) and undistorts the frames that arrive later with the new one: the per-call chain with each frame
    undistorted under the K in force when it arrived."""
    sizes = [(370, 1226), (240, 321)]
    models = ["plumb_4", "kitti_like_5"]
    Ks = [_K_for(s, k + 1) for k, s in enumerate(sizes)]
    raw = [synth.render_sequence("kitti", 9, seed=640 + k, width=c, height=r, K=Ks[k])["frames"] for k, (r, c) in enumerate(sizes)]
    vb = VOBatch(2, *SLOT, np.stack(Ks), OPT, frame_size=sizes, dist_coeffs=[_d8(m) for m in models], **CAPS)
    ref, K_at = [], [[Ks[s]] * 9 for s in range(2)]
    for s in range(2):
        st = initial_state(Ks[s], OPT, *match_bootstrap_frames(_und(raw[s][0], Ks[s], models[s]), _und(raw[s][2], Ks[s], models[s]),
                                                               OPT["feature_ratio"]))
        ref.append({k: st[k] for k in STATE_KEYS})
        vb.load(s, raw[s][2], ref[s])
    rng = np.random.default_rng(3)
    changed, live = False, [True, True]
    for f in range(3, 9):
        if f == 5:     # a new K for sequence 0 only, between two steps
            K2 = Ks[0] + np.array([[4.0, 0, 2.5], [0, 4.0, -1.75], [0, 0, 0]])
            vb.set_intrinsics([0], K2[None])
            assert vb.read_state(0)["status"] == VOBatch.OK
            for g in range(f, 9):
                K_at[0][g] = K2
        r = _copy(vb.step(_slot_layout([fr[f] for fr in raw], rng)))
        for s in range(2):
            if not live[s]:
                assert r["status"][s] != VOBatch.OK
                continue
            Kp, Kf = K_at[s][f - 1], K_at[s][f]
            prev, img = _und(raw[s][f - 1], Kp, models[s]), _und(raw[s][f], Kf, models[s])
            code, n_inl, host, new = _percall_step(ref[s], prev, img, Kf, r["pose_cw"][s].copy(), OPT)
            assert r["status"][s] == code and r["n_inliers"][s] == n_inl, (s, f)
            if code != VOBatch.OK:
                live[s] = False
                continue
            assert np.abs(r["pose_cw"][s] - host).max() <= 1e-12, (s, f)
            _assert_state(vb.read_state(s), new)
            ref[s] = new
            changed = changed or not np.array_equal(Kp, Kf)
    assert changed and live[0], "the sequence whose K changed must run every step for the comparison to mean much"
    vb.close()
