"""Per-sequence frame sizes against the C oracle: every batched tracker instance, the batched detector, the bootstrap's size
groups and the loop, at the sizes where their kernels branch (one-level images, widths under one pyramid tile or one detector
warp, heights under the border ring, odd level sizes) and with every window kind the tracker has: the staged <15,15> and
<21,21> kernels and the generic one, each with and without the per-sequence extent table.

The tracker and the detector are compared with `oracle` on each sequence's own tight image, in a batch of mixed sizes (the
extent table) and in a batch of one whose slot is the sequence's size (no table).  The bootstrap and the loop are compared
with the host chain and the per-call data flow."""
import numpy as np
import pytest

import oracle
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT, rodrigues
from monocular_visual_odometry_va4mr_b200 import _lib, cv2_compat, hotpath, synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch, initial_state, match_bootstrap_frames

SLOT = (376, 1242)        # rows, cols: the largest KITTI frame
VO_BORDER = 32            # internal.cuh: the REFLECT_101 ring around every pyramid level

# (rows, cols) of the sequences of a batch with a SLOT slot, and the edge each one targets.  Entries not larger than a
# window are left out for that window; sizes_for() adds the window's own minimal sizes.
SIZE_TABLE = [
    (376, 1242),   # the slot itself
    (376, 1241),   # KITTI 00-02
    (375, 1242),   # KITTI 03
    (370, 1226),   # KITTI 04-12
    (353, 1025),   # odd at every level in both dimensions (353 -> 177 -> 89 -> 45 -> 23); one column past eight 128-pixel tiles
    (257, 513),    # odd at every level in both dimensions down to 9 x 17, the sixth level of (5, 7)
    (240, 320),    # 4 levels with (15, 15) and (21, 21)
    (120, 640),    # 4 levels with (9, 13), 5 with (5, 7)
    (97, 161),     # 3 levels with (15, 15) and (21, 21); one 128-pixel tile and a 33-column tail
    (61, 129),     # 2 levels with (21, 21), level 1 of 31 rows under VO_BORDER + 2; one column past a 128-pixel tile
    (33, 383),     # 33 rows: level 0 under VO_BORDER + 2, the border ring bounces more than once
    (17, 129),     # 17 rows: one past a 16-row pyramid tile; 129: one column past a 128-pixel tile
    (45, 33),      # 33 columns: w & ~31 == 32, one column on the detector's unfused side
    (33, 31),      # 31 columns: w & ~31 == 0, every column on the unfused side
    (40, 29),      # 29 columns: narrower than the detector's 30-column warp
    (16, 16),      # one level with (15, 15), two with (5, 7)
    (23, 10),      # 10 columns: only the (5, 7) window is smaller
]
KITTI_WIDTHS = (1241, 1242, 1226)
TARGET_WIDTHS = (31, 33, 129, 161, 383, 1025) + KITTI_WIDTHS


def sizes_for(win):
    """the sizes of SIZE_TABLE legal for the window (w, h), then its smallest legal size and the slot's edges at that size"""
    ww, wh = win
    out = [s for s in SIZE_TABLE if s[0] > wh and s[1] > ww]
    out += [(wh + 1, ww + 1),      # the smallest legal size (batch.cu: a size must exceed the window): one pyramid level
            (wh + 1, SLOT[1]),     # full width, minimal height
            (SLOT[0], ww + 1)]     # full height, minimal width
    return out


# (window (w, h), maxLevel, criteria): the three criteria types, maxLevel 0 and above the slot's level count, every kernel
TRACK_CASES = [
    ((15, 15), 5, (3, 50, 0.01)),     # the reference options: klt_kernel_v3<15,15>
    ((15, 15), 0, (1, 20, 0.01)),     # one level, iteration count only
    ((21, 21), 3, (3, 30, 0.01)),     # klt_kernel_v3<21,21>
    ((21, 21), 8, (2, 30, 0.03)),     # maxLevel above the slot's 5 levels, eps only
    ((9, 13), 4, (3, 20, 0.001)),     # the generic klt_kernel from here on
    ((31, 31), 6, (1, 30, 0.01)),     # the largest window under VO_BORDER; the slot has 4 levels
    ((5, 7), 10, (3, 40, 0.01)),      # the slot has 6 levels
]


def _levels(size, win, max_level):
    return oracle.pyr_levels(size[1], size[0], win, max_level)


def _level_sizes(size, n):
    r, c = size
    out = []
    for _ in range(n):
        out.append((r, c))
        r, c = (r + 1) // 2, (c + 1) // 2
    return out


# ---------------------------------------------------------------------------------------------------- the table itself (CPU)
def test_size_table_covers_its_edges():
    """What the comments of SIZE_TABLE and sizes_for claim, checked with the oracle's level count and plain arithmetic."""
    # the level counts of the issue-style table: size -> {(window, maxLevel): levels}
    want = {(16, 16): {((15, 15), 5): 1, ((5, 7), 10): 2}, (33, 31): {((15, 15), 5): 2, ((21, 21), 3): 1, ((5, 7), 10): 3},
            (97, 161): {((15, 15), 5): 3, ((21, 21), 3): 3, ((5, 7), 10): 4},
            (240, 320): {((15, 15), 5): 4, ((21, 21), 3): 4, ((5, 7), 10): 6},
            (376, 1242): {((15, 15), 5): 5, ((21, 21), 3): 4, ((5, 7), 10): 6}}
    for size, cases in want.items():
        for (win, ml), n in cases.items():
            assert _levels(size, win, ml) == n, (size, win, ml)
    assert len(set(SIZE_TABLE)) == len(SIZE_TABLE)
    for win, ml, crit in TRACK_CASES:
        ww, wh = win
        assert ww < VO_BORDER and wh < VO_BORDER
        sizes = sizes_for(win)
        assert all(wh < r <= SLOT[0] and ww < c <= SLOT[1] for r, c in sizes), win
        assert SLOT in sizes and (SLOT[0], ww + 1) in sizes and (wh + 1, SLOT[1]) in sizes
        assert _levels((wh + 1, ww + 1), win, ml) == 1 and (wh + 1, ww + 1) in sizes
        # every level count from 1 to the slot's
        n_slot = _levels(SLOT, win, ml)
        assert {_levels(s, win, ml) for s in sizes} == set(range(1, n_slot + 1)), (win, ml)
        # at every level of the slot some sequence has an odd height there, and one under VO_BORDER + 2
        for lvl in range(n_slot):
            hs = [_level_sizes(s, _levels(s, win, ml))[lvl][0] for s in sizes if _levels(s, win, ml) > lvl]
            assert any(h % 2 for h in hs), (win, ml, lvl)
        assert any(r < VO_BORDER + 2 for r, _ in sizes), win
        # the widths where the pyramid and the detector branch, wherever the window allows them
        widths = {c for _, c in sizes}
        for w in TARGET_WIDTHS:
            assert w <= ww or w in widths, (win, w)
        if ww < 29:
            assert any(c < 30 for c in widths), win                       # narrower than the detector's warp
        if ww < 16:
            assert any(r == 17 for r, _ in sizes), win                    # one row past a 16-row tile
        assert any(c < 128 for c in widths) and any(128 < c < 256 for c in widths)
    assert (31 & ~31) == 0 and (33 & ~31) == 32
    # the cases cover maxLevel 0, a maxLevel above the slot's level count, the three criteria types and every kernel kind
    assert any(ml == 0 for _, ml, _ in TRACK_CASES)
    assert any(ml >= _levels(SLOT, win, ml) for win, ml, _ in TRACK_CASES if ml)
    assert {crit[0] for _, _, crit in TRACK_CASES} == {1, 2, 3}
    assert {(15, 15), (21, 21)} <= {w for w, _, _ in TRACK_CASES}
    assert len({w for w, _, _ in TRACK_CASES} - {(15, 15), (21, 21)}) >= 3


# ---------------------------------------------------------------------------------------------------- shared inputs
@pytest.fixture(scope="module")
def slot_frames():
    """Three consecutive KITTI frames at the slot size; a sequence's image is a crop of them."""
    return synth.render_sequence("kitti", 3, seed=910, width=SLOT[1], height=SLOT[0])["frames"]


def _crops(frames, sizes, rng):
    """per sequence: the frames cropped to its size at a random offset (the crop moves with the scene)"""
    out = []
    for r, c in sizes:
        y0, x0 = int(rng.integers(0, SLOT[0] - r + 1)), int(rng.integers(0, SLOT[1] - c + 1))
        out.append(np.ascontiguousarray(frames[:, y0:y0 + r, x0:x0 + c]))
    return out


def _slot_layout(images, rng, slot=SLOT):
    """per-sequence images as the top-left of slot-sized frames whose other bytes are random"""
    out = rng.integers(0, 256, (len(images),) + slot, dtype=np.uint8)
    for k, im in enumerate(images):
        out[k, :im.shape[0], :im.shape[1]] = im
    return out


def _edge_offsets(hw, w):
    """level coordinates near the low edge (0) of a level for a window of w = 2 hw + 1 taps: the window's first tap just
    past -w (lost), just inside it, straddling the edge, at it, and inside the image"""
    return np.float32([-w + hw - 0.6, -w + hw + 0.3, -hw - 0.45, -1.2, -0.3, 0.0, 0.7, hw - 0.5, hw + 0.5, hw + 2.25])


def _track_points(size, win, n_levels, rng):
    """windows straddling, inside and just outside each of the four edges of the image at every level and at its four
    corners, points well outside, on a quarter-pixel grid, offset by 3.2e-5 (a negative bilinear weight) and inside"""
    r, c = size
    hx, hy = (win[0] - 1) / 2, (win[1] - 1) / 2
    pts = []
    for lvl in range(n_levels + 1):
        s = float(1 << lvl)
        wl, hl = -(-c // (1 << lvl)), -(-r // (1 << lvl))
        ox, oy = _edge_offsets(hx, win[0]), _edge_offsets(hy, win[1])
        lo_x, hi_x = ox, wl - 1 - ox
        lo_y, hi_y = oy, hl - 1 - oy
        for xs in (lo_x, hi_x):           # left and right edge
            for x in xs:
                pts.append((x * s, rng.uniform(0, r)))
        for ys in (lo_y, hi_y):           # top and bottom edge
            for y in ys:
                pts.append((rng.uniform(0, c), y * s))
        for xs in (lo_x, hi_x):           # the four corners
            for ys in (lo_y, hi_y):
                for i in (0, 2, 4, 7, 9):
                    pts.append((xs[i] * s, ys[i] * s))
    pts = np.float32(pts)
    far = np.float32([(-500, r / 2), (c + 500, r / 2), (c / 2, -400), (c / 2, r + 400), (-1e4, -1e4), (3 * c, 3 * r)])
    quarter = np.rint(np.column_stack([rng.uniform(-4, c + 4, 40), rng.uniform(-4, r + 4, 40)]) * 4) / 4
    neg = quarter[:30] + np.float32(3.2e-5)
    inner = np.column_stack([rng.uniform(0.2 * c, 0.8 * c, 60), rng.uniform(0.2 * r, 0.8 * r, 60)])
    return np.concatenate([pts, far, quarter, neg, inner]).astype(np.float32)


def _copy(r):
    return {k: np.array(v) for k, v in r.items()}


# ---------------------------------------------------------------------------------------------------- tracker
@pytest.mark.gpu
@pytest.mark.parametrize("win,max_level,crit", TRACK_CASES, ids=[f"{w[0]}x{w[1]}-L{m}-c{c[0]}" for w, m, c in TRACK_CASES])
def test_tracker_against_oracle(slot_frames, win, max_level, crit):
    rng = np.random.default_rng(win[0] * 100 + win[1] + max_level)
    sizes = sizes_for(win)
    crops = _crops(slot_frames, sizes, rng)
    n_lv = [_levels(s, win, max_level) for s in sizes]
    lm = [_track_points(s, win, n, rng) for s, n in zip(sizes, n_lv)]
    cand = [_track_points(s, win, n, rng)[::-1].copy() for s, n in zip(sizes, n_lv)]
    L, Cn = max(len(p) for p in lm), max(len(p) for p in cand)
    B = len(sizes)
    lm_pts, cand_pts = np.zeros((B, L, 2), np.float32), np.zeros((B, Cn, 2), np.float32)
    for k in range(B):
        lm_pts[k, :len(lm[k])], cand_pts[k, :len(cand[k])] = lm[k], cand[k]
    lm_obj = np.zeros((B, L, 3), np.float32)
    lm_obj[..., 2] = 10.0
    n_lm = np.int32([len(p) for p in lm])
    n_cand = np.int32([len(p) for p in cand])
    kw = dict(win=win, max_level=max_level, criteria=crit, max_landmarks=L, max_candidates=Cn)

    mixed = SequenceBatch(B, *SLOT, synth.K_KITTI, frame_size=sizes, **kw)
    mixed.prime(_slot_layout([c[0] for c in crops], rng))
    got_mixed = [_copy(mixed.step(_slot_layout([c[f] for c in crops], rng), lm_pts, lm_obj, n_lm, cand_pts, n_cand)) for f in (1, 2)]
    mixed.close()

    outcomes = set()
    for k, (size, im) in enumerate(zip(sizes, crops)):
        one = SequenceBatch(1, *size, synth.K_KITTI, **kw)
        one.prime(im[0][None])
        got_one = [_copy(one.step(im[f][None].copy(), lm_pts[k:k + 1].copy(), lm_obj[k:k + 1].copy(), n_lm[k:k + 1].copy(),
                                  cand_pts[k:k + 1].copy(), n_cand[k:k + 1].copy())) for f in (1, 2)]
        one.close()
        for f in (1, 2):
            for key, pts in (("lm", lm[k]), ("cand", cand[k])):
                n = len(pts)
                rp, rst, _ = oracle.calc_optical_flow_pyr_lk(im[f - 1], im[f], pts, win, max_level, crit)
                cp, cst, _ = cv2_compat.calcOpticalFlowPyrLK(im[f - 1], im[f], pts, None, winSize=win, maxLevel=max_level, criteria=crit)
                rst, ok = rst.ravel(), rst.ravel() == 1
                assert np.array_equal(cst.ravel(), rst), (size, f, key)
                for name, got in (("mixed", got_mixed[f - 1]), ("one", got_one[f - 1])):
                    row = 0 if name == "one" else k
                    nxt, st = got[f"{key}_next"][row, :n], got[f"{key}_status"][row, :n]
                    assert np.array_equal(st, rst), (name, size, f, key, np.flatnonzero(st != rst)[:8])
                    assert np.array_equal(nxt[ok], rp[ok]), (name, size, f, key)
                    assert np.array_equal(nxt, cp.reshape(-1, 2)), (name, size, f, key)
                outcomes |= set(rst.tolist())
    assert outcomes == {0, 1}       # both outcomes are compared


# ---------------------------------------------------------------------------------------------------- detector
def _corner_images(crops, rng):
    """level-0 images of the detector batch: synthetic frames, strong corners on the first and last rows and columns, a
    fine checkerboard patch (tied maxima), a flat image"""
    out = []
    for k, im in enumerate(crops):
        r, c = im.shape
        kind = k % 4
        if kind == 0:
            out.append(im.copy())
        elif kind == 1:
            # spikes on the first two and last two rows and columns: cv2 never returns the outermost ones, the next ones win
            a = rng.integers(90, 120, (r, c), dtype=np.uint8)
            for x in range(0, c, 4):
                a[(x // 4) % 2, x] = a[r - 1 - (x // 4) % 2, x] = 255
            for y in range(0, r, 4):
                a[y, (y // 4) % 2] = a[y, c - 1 - (y // 4) % 2] = 0
            out.append(a)
        elif kind == 2:
            # across the column w & ~31 where the detector's row filter changes from fused to unfused arithmetic, which
            # breaks some ties one way on one side and the other way on the other
            a = im.copy()
            ph, pw = min(r, 48), min(c, 64)
            y0, x0 = (r - ph) // 2, min(max((c & ~31) - pw // 2, 0), c - pw)
            yy, xx = np.mgrid[:ph, :pw]
            a[y0:y0 + ph, x0:x0 + pw] = np.where(((yy // 2) + (xx // 2)) % 2 == 0, 40, 215).astype(np.uint8)
            out.append(a)
        else:
            out.append(np.full((r, c), 77, np.uint8))
    return out


# (max_corners, quality, min_dist, slot): min_dist <= 5 needs a smaller slot (the cell grid lives in shared memory)
GFTT_CASES = [
    (1400, 0.1, 10.0, SLOT),
    (25, 0.01, 25.0, SLOT),
    (7, 0.3, 10.0, SLOT),
    (300, 0.05, 3.0, (240, 320)),
    (5000, 0.02, 1.0, (97, 129)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("max_corners,quality,min_dist,slot", GFTT_CASES)
def test_detector_against_oracle(slot_frames, max_corners, quality, min_dist, slot):
    rng = np.random.default_rng(int(min_dist * 1000 + max_corners))
    sizes = [s for s in sizes_for((5, 7)) if s[0] <= slot[0] and s[1] <= slot[1]]
    sizes += [slot] * (slot not in sizes)
    images = _corner_images([c[0] for c in _crops(slot_frames, sizes, rng)], rng)
    layout = _slot_layout(images, rng, slot)
    for k, (r, c) in enumerate(sizes):    # strong corners in every slot's random padding: never returned
        layout[k, r + 2:r + 9:3, ::5] = 255
        layout[k, ::4, c + 2:c + 9:3] = 255
        layout[k, r + 1:r + 6, c + 1:c + 6] = 255
    sb = SequenceBatch(len(sizes), *slot, synth.K_KITTI, win=(5, 7), max_landmarks=4, max_candidates=0, frame_size=sizes)
    sb.prime(layout)
    corners, n = sb.good_features(max_corners, quality, min_dist)
    sb.close()
    found = 0
    for k, (size, im) in enumerate(zip(sizes, images)):
        want = oracle.good_features_to_track(im, max_corners, quality, min_dist)
        want = np.zeros((0, 2), np.float32) if want is None else want.reshape(-1, 2)
        assert n[k] == len(want), (size, k % 4, n[k], len(want))
        assert np.array_equal(corners[k, :n[k]], want), (size, k % 4)
        found += n[k]
    assert found > 0 and n[2::4].all()


@pytest.mark.gpu
def test_detector_refuses_a_cell_grid_beyond_shared_memory():
    sb = SequenceBatch(2, *SLOT, synth.K_KITTI, max_landmarks=4, max_candidates=0, frame_size=[SLOT, (33, 31)])
    sb.prime(np.zeros((2,) + SLOT, np.uint8))
    with pytest.raises(_lib.B200VOError):
        sb.good_features(1400, 0.1, 3.0)
    sb.close()


# ---------------------------------------------------------------------------------------------------- bootstrap
CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")


def _K(f, rows, cols):
    return np.array([[f, 0.0, cols / 2 - 0.5], [0.0, f, rows / 2 + 3.25], [0.0, 0.0, 1.0]])


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def _host_chain(K, f0, f1, options=OPT):
    """the host bootstrap chain; None where it raises (too few matches or no essential matrix)"""
    try:
        return initial_state(K, options, *match_bootstrap_frames(f0, f1, options["feature_ratio"]))
    except Exception:
        return None


@pytest.mark.gpu
def test_bootstrap_interleaved_sizes():
    A, B, C, D = (376, 1241), (370, 1226), (240, 320), (33, 31)
    # the KITTI 00-02 group fills two SIFT chunks; the groups are interleaved by index; D is too small for SIFT
    layout = [A, B, C, A, D, A, B, A, C, A, B, A, A, A, A, A, A, A, A, A]
    assert layout.count(A) >= 14
    Ks = {A: synth.K_KITTI, B: _K(707.0912, *B), C: _K(300.0, *C), D: _K(40.0, *D)}
    seqs = []
    for i, size in enumerate(layout):
        fr = synth.render_sequence("kitti", 5, seed=500 + i, width=size[1], height=size[0], K=Ks[size])["frames"]
        seqs.append((fr, Ks[size], size))
    K = np.stack([K for _, K, _ in seqs])
    sizes = [s for _, _, s in seqs]
    dev = VOBatch(len(seqs), *SLOT, K, OPT, frame_size=sizes, **CAPS)
    host = VOBatch(len(seqs), *SLOT, K, OPT, frame_size=sizes, **CAPS)
    r = _copy(dev.bootstrap([fr[0] for fr, _, _ in seqs], [fr[2] for fr, _, _ in seqs]))
    ok = []
    for s, (fr, Ks_, size) in enumerate(seqs):
        st = _host_chain(Ks_, fr[0], fr[2])
        if st is None:
            assert r["status"][s] == VOBatch.NO_BOOTSTRAP and r["num_pts"][s] == 0, s
            assert dev.read_state(s)["status"] == VOBatch.NO_BOOTSTRAP
            continue
        assert r["status"][s] == VOBatch.OK and r["num_pts"][s] == st["num_pts"], s
        assert r["n_lm"][s] == len(st["lm"]) and r["n_cand"][s] == len(st["keys"]), s
        _assert_state(dev.read_state(s), st)
        host.load(s, fr[2], st)
        ok.append(s)
    assert r["status"][layout.index(D)] == VOBatch.NO_BOOTSTRAP
    assert {layout[s] for s in ok} == {A, B, C} and len(ok) >= len(layout) - 3
    # the resident frame is the second bootstrap frame at the sequence's own size
    rd, rh = _copy(dev.step([fr[3] for fr, _, _ in seqs])), _copy(host.step([fr[3] for fr, _, _ in seqs]))
    for k in rd:
        assert np.array_equal(rd[k][ok], rh[k][ok]), k

    # a subset in non-monotone index order, mixing every size group: again the host chain, on frames 1 and 4
    listed = [11, 2, 4, 0, 8, 6, 19]
    r = _copy(dev.bootstrap([seqs[s][0][1] for s in listed], [seqs[s][0][4] for s in listed], seqs=listed))
    for k, s in enumerate(listed):
        fr, Ks_, _ = seqs[s]
        st = _host_chain(Ks_, fr[1], fr[4])
        if st is None:
            assert r["status"][k] == VOBatch.NO_BOOTSTRAP and dev.read_state(s)["status"] == VOBatch.NO_BOOTSTRAP, s
            continue
        assert r["status"][k] == VOBatch.OK and r["num_pts"][k] == st["num_pts"], s
        assert r["n_lm"][k] == len(st["lm"]) and r["n_cand"][k] == len(st["keys"]), s
        _assert_state(dev.read_state(s), st)
    assert r["status"][listed.index(4)] == VOBatch.NO_BOOTSTRAP
    assert (r["status"] == VOBatch.OK).sum() >= len(listed) - 2
    others = [s for s in range(len(seqs)) if s not in listed]
    for s in others:            # untouched: as the twin that never got the call
        a, b = dev.read_state(s), host.read_state(s)
        _assert_state(a, b)
        assert a["status"] == (b["status"] if s in ok else VOBatch.NO_BOOTSTRAP), s
    dev.close()
    host.close()


# ---------------------------------------------------------------------------------------------------- the loop, (21, 21)
OPT21 = dict(OPT, winSize=(21, 21), maxLevel=3)


def _percall_step(st, prev, img, K, pose_cw, o):
    """MiniVO.step on the per-call entry points with the options `o` (test_vo_loop_gpu.py).  Returns (status, n_inliers,
    host pose (12,), new state); the new pose of the state is `pose_cw` (the loop's), so that an ulp of sin / cos does not
    accumulate."""
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


@pytest.mark.gpu
def test_loop_21x21_mixed_sizes_equals_per_call_path():
    sizes = [(376, 1241), (375, 1242), (370, 1226), (353, 1025), (376, 1241), (300, 900)]
    seqs = []
    for i, size in enumerate(sizes):
        K = synth.K_KITTI if size[1] >= 1241 else _K(650.0, *size)
        fr = synth.render_sequence("kitti", 13, seed=700 + i, width=size[1], height=size[0], K=K)["frames"]
        st = initial_state(K, OPT21, *match_bootstrap_frames(fr[0], fr[2], OPT21["feature_ratio"]))
        seqs.append((fr, K, st))
    vb = VOBatch(len(seqs), *SLOT, np.stack([K for _, K, _ in seqs]), OPT21, frame_size=sizes, **CAPS)
    for s, (fr, _, st) in enumerate(seqs):
        vb.load(s, fr[2], st)
    ref = [dict((k, st[k]) for k in STATE_KEYS) for _, _, st in seqs]
    live = [True] * len(seqs)
    for f in range(3, 13):
        r = vb.step([fr[f] for fr, _, _ in seqs])
        for s, (frames, K, _) in enumerate(seqs):
            if not live[s]:
                assert r["status"][s] != VOBatch.OK
                continue
            code, n_inl, host, new = _percall_step(ref[s], frames[f - 1], frames[f], K, r["pose_cw"][s].copy(), OPT21)
            assert r["status"][s] == code, (s, f)
            assert r["n_inliers"][s] == n_inl, (s, f)
            if code != VOBatch.OK:
                live[s] = False
                continue
            assert np.abs(r["pose_cw"][s] - host).max() <= 1e-12, (s, f)
            assert r["n_lm"][s] == len(new["lm"]) and r["n_cand"][s] == len(new["keys"]), (s, f)
            _assert_state(vb.read_state(s), new)
            ref[s] = new
    vb.close()
    assert sum(live) >= 4, "too few sequences ran all 10 steps for the comparison to mean much"
