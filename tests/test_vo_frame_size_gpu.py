"""Per-sequence frame sizes (VOBatch / SequenceBatch `frame_size`, `set_frame_size`): the constructor's rows x cols is the slot,
each sequence's image is the top-left of its slot, and a sequence in a batch of mixed sizes must compute exactly what it
computes in a batch of its own size -- whatever the bytes outside its image hold."""
import numpy as np
import pytest

from mini_vo import REFERENCE_KITTI_OPTIONS as OPT
from monocular_visual_odometry_va4mr_b200 import _lib, cv2_compat, synth
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch, VOBatch

pytestmark = pytest.mark.gpu

CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
N_FRAMES = 15
SLOT = (376, 1242)


def _K(fx, fy, cx, cy):
    return np.array([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]])


# the three KITTI odometry groups (00-02, 03, 04-12): calibration and native image size (rows, cols)
KITTI = [(_K(718.856, 718.856, 607.1928, 185.2157), (376, 1241)), (_K(721.5377, 721.5377, 609.5593, 172.854), (375, 1242)),
         (_K(707.0912, 707.0912, 601.8873, 183.1104), (370, 1226))]


@pytest.fixture(scope="module")
def scenes():
    """Six sequences, two per KITTI group, each rendered at its size through its calibration."""
    out = []
    for i in range(6):
        K, (r, c) = KITTI[i // 2]
        s = synth.render_sequence("kitti", N_FRAMES, seed=300 + i, width=c, height=r, K=K)
        out.append((s["frames"], K, (r, c)))
    return out


def _copy(r):
    return {k: np.array(v) for k, v in r.items()}


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k
    assert got["status"] == want["status"]


def _slot_frames(images, fill, rng):
    """per-sequence images in the slot layout, the bytes outside each image set to `fill` ('zero' or 'random')"""
    out = np.zeros((len(images),) + SLOT, np.uint8) if fill == "zero" else rng.integers(0, 256, (len(images),) + SLOT, dtype=np.uint8)
    for k, im in enumerate(images):
        out[k, :im.shape[0], :im.shape[1]] = im
    return out


def _mixed_run(scenes, fill=None, seed=0):
    """One VOBatch of the six sequences in 1242 x 376 slots: device bootstrap on frames 0 and 2, then 12 steps.
    fill None: frames handed over as lists of per-sequence images; else slot-layout arrays with that padding."""
    rng = np.random.default_rng(seed)
    vb = VOBatch(len(scenes), *SLOT, np.stack([K for _, K, _ in scenes]), OPT, frame_size=[sz for _, _, sz in scenes], **CAPS)
    frames = lambda f: [fr[f] for fr, _, _ in scenes] if fill is None else _slot_frames([fr[f] for fr, _, _ in scenes], fill, rng)
    boot = _copy(vb.bootstrap(frames(0), frames(2)))
    states0 = [vb.read_state(s) for s in range(len(scenes))]
    steps = []
    for f in range(3, N_FRAMES):
        r = _copy(vb.step(frames(f)))
        steps.append((r, [vb.read_state(s) for s in range(len(scenes))]))
    vb.close()
    return boot, states0, steps


@pytest.fixture(scope="module")
def mixed_run(scenes):
    return _mixed_run(scenes)


def _run_one(frames, K, size, n_steps=N_FRAMES - 3, slot=None, frame_size=None):
    one = VOBatch(1, *(slot or size), K, OPT, frame_size=frame_size, **CAPS)
    boot = _copy(one.bootstrap([frames[0]], [frames[2]]) if frame_size is not None else one.bootstrap(frames[0][None], frames[2][None]))
    states0 = one.read_state(0)
    steps = []
    for f in range(3, 3 + n_steps):
        r = _copy(one.step([frames[f]]) if frame_size is not None else one.step(frames[f][None]))
        steps.append((r, one.read_state(0)))
    one.close()
    return boot, states0, steps


def test_mixed_batch_equals_batches_of_one(scenes, mixed_run):
    boot, states0, steps = mixed_run
    assert list(boot["status"]) == [VOBatch.OK] * len(scenes)
    for s, (frames, K, size) in enumerate(scenes):
        b1, st1, steps1 = _run_one(frames, K, size)
        for k in b1:
            assert b1[k][0] == boot[k][s], (s, k)
        _assert_state(st1, states0[s])
        for i, (r1, got) in enumerate(steps1):
            r, states = steps[i]
            for k in r1:
                assert np.array_equal(r1[k][0], r[k][s]), (s, i, k)
            _assert_state(got, states[s])
    # the sequences keep tracking: the comparison covers live steps
    assert (steps[-1][0]["status"] == VOBatch.OK).sum() >= 4


def _assert_runs_equal(a, b):
    boot_a, st_a, steps_a = a
    boot_b, st_b, steps_b = b
    for k in boot_a:
        assert np.array_equal(boot_a[k], boot_b[k]), k
    for x, y in zip(st_a, st_b):
        _assert_state(x, y)
    for (ra, sa), (rb, sb) in zip(steps_a, steps_b):
        for k in ra:
            assert np.array_equal(ra[k], rb[k]), k
        for x, y in zip(sa, sb):
            _assert_state(x, y)


def test_padding_is_never_read(scenes, mixed_run):
    noisy = _mixed_run(scenes, "random", seed=1)
    _assert_runs_equal(noisy, _mixed_run(scenes, "zero"))
    _assert_runs_equal(noisy, mixed_run)


def test_shrunk_slot_reads_no_stale_bytes(scenes):
    """A slot that held a full-size sequence is shrunk and bootstrapped again: the new sequence must equal a fresh batch of one."""
    big = synth.render_sequence("kitti", 6, seed=77, width=SLOT[1], height=SLOT[0], K=KITTI[0][0])["frames"]
    frames, K, size = scenes[4]
    vb = VOBatch(2, *SLOT, KITTI[0][0], OPT, **CAPS)
    assert list(vb.bootstrap(np.stack([big[0], big[0]]), np.stack([big[2], big[2]]))["status"]) == [VOBatch.OK] * 2
    for f in range(3, 6):
        vb.step(np.stack([big[f], big[f]]))
    vb.set_frame_size([0], [size])
    assert vb.read_state(0)["status"] == VOBatch.IDLE and vb.read_state(1)["status"] == VOBatch.OK
    vb.set_intrinsics([0], K[None])
    boot = _copy(vb.bootstrap([frames[0]], [frames[2]], seqs=[0]))
    st0 = vb.read_state(0)
    n = 6
    steps = []
    for f in range(3, 3 + n):
        steps.append((_copy(vb.step([frames[f], big[min(f, 5)]])), vb.read_state(0)))
    vb.close()
    b1, st1, steps1 = _run_one(frames, K, size, n)
    for k in b1:
        assert b1[k][0] == boot[k][0], k
    _assert_state(st1, st0)
    for (r1, s1), (r, s) in zip(steps1, steps):
        for k in r1:
            assert np.array_equal(r1[k][0], r[k][0]), k
        _assert_state(s1, s)


def test_fewer_levels_than_the_slot():
    """1241 x 376 has 5 pyramid levels with the reference options, a 1241 x 768 slot 6."""
    K, size = KITTI[0]
    frames = synth.render_sequence("kitti", 10, seed=41, width=size[1], height=size[0], K=K)["frames"]
    a = _run_one(frames, K, size, 7, slot=(768, 1241), frame_size=[size])
    b = _run_one(frames, K, size, 7)
    assert a[0]["status"][0] == VOBatch.OK
    _assert_runs_equal((a[0], [a[1]], [(r, [s]) for r, s in a[2]]), (b[0], [b[1]], [(r, [s]) for r, s in b[2]]))


def _edge_points(size, n_lm, rng):
    """points near the sequence's right and bottom edge at every pyramid level: inside, straddling and outside its image
    (but inside the slot), plus interior ones so that the pose has landmarks to use"""
    r, c = size
    pts = []
    for lvl in range(6):
        s = 1 << lvl
        wl, hl = -(-c // s), -(-r // s)
        for d in (-9.3, -4.5, -1.2, 0.4, 2.7, 6.1, 13.8):
            pts.append(((wl + d) * s, rng.uniform(20, r - 20)))
            pts.append((rng.uniform(20, c - 20), (hl + d) * s))
            pts.append(((wl + d) * s, (hl + d) * s))
    pts = np.float32(pts)
    inner = np.stack([rng.uniform(30, c - 30, n_lm - len(pts)), rng.uniform(30, r - 30, n_lm - len(pts))], 1).astype(np.float32)
    return np.concatenate([pts, inner])


def test_sequence_batch_edges_and_corners(scenes):
    rng = np.random.default_rng(5)
    seqs = [scenes[0], scenes[2], scenes[4]]
    n_lm, L, Cn = 300, 320, 320
    sizes = [sz for _, _, sz in seqs]
    sb = SequenceBatch(len(seqs), *SLOT, np.stack([K for _, K, _ in seqs]), max_landmarks=L, max_candidates=Cn, frame_size=sizes)
    lm_pts = np.zeros((len(seqs), L, 2), np.float32)
    lm_obj = np.zeros((len(seqs), L, 3), np.float32)
    cand = np.zeros((len(seqs), Cn, 2), np.float32)
    for k, (fr, K, size) in enumerate(seqs):
        lm_pts[k, :n_lm] = _edge_points(size, n_lm, rng)
        lm_obj[k, :n_lm] = np.c_[rng.uniform(-5, 5, (n_lm, 2)), rng.uniform(8, 40, n_lm)]
        cand[k, :n_lm] = _edge_points(size, n_lm, rng)[::-1]
    n = np.full(len(seqs), n_lm, np.int32)
    # a strong corner in every slot's padding (right of and below the image): it must never be detected
    images = lambda f: [fr[f] for fr, _, _ in seqs]
    prime = _slot_frames(images(0), "zero", rng)
    for k, (r, c) in enumerate(sizes):
        if c < SLOT[1]:
            prime[k, 100:120, c:] = 255
        if r < SLOT[0]:
            prime[k, r:, 300:320] = 255
    sb.prime(prime)
    corners, nc = sb.good_features(1400, 0.1, 10.0)
    for k, (fr, _, (r, c)) in enumerate(seqs):
        want = cv2_compat.goodFeaturesToTrack(fr[0], 1400, 0.1, 10, blockSize=3, useHarrisDetector=False, mask=None).reshape(-1, 2)
        assert nc[k] == len(want) and np.array_equal(corners[k, :nc[k]], want), k
    out = _copy(sb.step(images(1), lm_pts, lm_obj, n, cand, n))
    sb.close()
    for k, (fr, K, size) in enumerate(seqs):
        one = SequenceBatch(1, *size, K, max_landmarks=L, max_candidates=Cn)
        one.prime(fr[0][None])
        c1, n1 = one.good_features(1400, 0.1, 10.0)
        assert n1[0] == nc[k] and np.array_equal(c1[0, :n1[0]], corners[k, :nc[k]])
        r1 = one.step(np.ascontiguousarray(fr[1][None]), lm_pts[k:k + 1].copy(), lm_obj[k:k + 1].copy(), n[k:k + 1].copy(),
                      cand[k:k + 1].copy(), n[k:k + 1].copy())
        for key in ("lm_next", "lm_status", "cand_next", "cand_status", "pose", "pnp_ok", "inlier_mask", "n_inliers"):
            assert np.array_equal(r1[key][0], out[key][k], equal_nan=True), (k, key)
        st = out["lm_status"][k, :n_lm]
        assert 0 < st.sum() < n_lm, k    # some edge points are lost, the interior ones track
        one.close()


def _refusals(obj, fn_name):
    """every refused set_frame_size argument: ValueError through Python, B200VO_E_BADARG through the C ABI"""
    b = obj.batch
    bad = [([b], [(300, 1000)]), ([-1], [(300, 1000)]), ([0, 0], [(300, 1000), (300, 1000)]), ([], np.zeros((0, 2), int)),
           ([0], [(SLOT[0] + 1, 1000)]), ([0], [(300, SLOT[1] + 1)]), ([0], [(15, 1000)]), ([0], [(300, 15)]), ([0], [(300.5, 1000)]),
           ([0, 1], [(300, 1000)])]
    for seqs, sizes in bad:
        with pytest.raises(ValueError):
            obj.set_frame_size(seqs, sizes)
    fn = getattr(obj.ctx.lib, fn_name)
    one = np.int32([300])
    assert fn(obj.h, 1, None, one.ctypes.data_as(_lib.c_i32p), one.ctypes.data_as(_lib.c_i32p)) == -1
    assert fn(obj.h, 1, np.int32([0]).ctypes.data_as(_lib.c_i32p), None, one.ctypes.data_as(_lib.c_i32p)) == -1
    assert fn(obj.h, 1, np.int32([0]).ctypes.data_as(_lib.c_i32p), one.ctypes.data_as(_lib.c_i32p), None) == -1


def test_validation(scenes):
    frames, K, size = scenes[0]
    vb = VOBatch(2, *SLOT, K, OPT, **CAPS)
    vb.bootstrap(np.stack([_slot_frames([frames[0]], "zero", None)[0]] * 2), np.stack([_slot_frames([frames[2]], "zero", None)[0]] * 2))
    before = [vb.read_state(s) for s in range(2)]
    launches = vb.ctx.launch_count()
    _refusals(vb, "b200vo_loop_set_frame_size")
    # submitted frames still waiting
    pf = vb.pinned_frames()
    pf[0] = _slot_frames([frames[3]] * 2, "zero", None)
    vb.submit_frames(pf[0])
    with pytest.raises(ValueError):
        vb.set_frame_size([0], [size])
    assert vb.ctx.launch_count() == launches
    for s in range(2):
        _assert_state(vb.read_state(s), before[s])
    assert list(vb.frame_size[:, 0]) == [SLOT[0]] * 2
    vb.step(None)
    # accepted: the listed sequence becomes IDLE and is skipped; the other one steps on
    vb.set_frame_size([1], [size])
    assert vb.read_state(1)["status"] == VOBatch.IDLE
    r = vb.step(_slot_frames([frames[4], frames[4]], "zero", None))
    assert r["status"][1] == VOBatch.IDLE and r["status"][0] == VOBatch.OK
    with pytest.raises(ValueError):
        vb.load(1, np.zeros(SLOT, np.uint8), before[1])   # the frame must have the sequence's size
    vb.close()

    sb = SequenceBatch(2, *SLOT, K, max_landmarks=64, max_candidates=64)
    sb.prime(np.zeros((2,) + SLOT, np.uint8))
    launches = sb.ctx.launch_count()
    _refusals(sb, "b200vo_batch_set_frame_size")
    assert sb.ctx.launch_count() == launches
    sb.set_frame_size([0], [size])
    z = np.zeros((2, 64, 2), np.float32)
    with pytest.raises(_lib.B200VOError):   # the resident pyramids were built at the old size: prime first
        sb.step(np.zeros((2,) + SLOT, np.uint8), z, np.zeros((2, 64, 3), np.float32), np.zeros(2, np.int32), z, np.zeros(2, np.int32))
    sb.prime(np.zeros((2,) + SLOT, np.uint8))
    sb.step(np.zeros((2,) + SLOT, np.uint8), z, np.zeros((2, 64, 3), np.float32), np.zeros(2, np.int32), z, np.zeros(2, np.int32))
    sb.close()
