"""Listed steps (VOBatch.step / step_dev / submit_frames / submit_frames_dev with `seqs`, b200vo_loop_*_seqs): a step that
advances only the sequences that have a new frame.  A listed sequence must compute exactly what it computes in a batch of
one fed only its own frames; a sequence that is not listed must not change at all, and must resume from its current frame."""
import ctypes as C

import numpy as np
import pytest

from mini_vo import REFERENCE_KITTI_OPTIONS as OPT
from monocular_visual_odometry_va4mr_b200 import synth
from monocular_visual_odometry_va4mr_b200._lib import c_i32p, c_u8p
from monocular_visual_odometry_va4mr_b200.batch import VOBatch

pytestmark = pytest.mark.gpu

CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
SLOT = (376, 1242)
N_SEQ, N_TICKS, LATE, LATE_TICK = 6, 14, 4, 6
RES_KEYS = ("status", "n_inliers", "n_lm", "n_cand", "pose_cw")


def _K(fx, fy, cx, cy):
    return np.array([[fx, 0.0, cx], [0.0, fy, cy], [0.0, 0.0, 1.0]])


# the three KITTI odometry groups (00-02, 03, 04-12): calibration and native image size (rows, cols)
KITTI = [(_K(718.856, 718.856, 607.1928, 185.2157), (376, 1241)), (_K(721.5377, 721.5377, 609.5593, 172.854), (375, 1242)),
         (_K(707.0912, 707.0912, 601.8873, 183.1104), (370, 1226))]


def _schedule():
    """The sequences that have a frame at each tick, in a non-monotone order: 0 every tick; 1 and 2 every other tick with
    different phases; 3 ends after 5 frames; 4 is bootstrapped at LATE_TICK and ticks from then on; 5 has a 4-tick gap."""
    rng = np.random.default_rng(7)
    out = []
    for t in range(N_TICKS):
        s = [0]
        s += [1] if t % 2 == 0 else [2]
        s += [3] if t < 5 else []
        s += [LATE] if t >= LATE_TICK else []
        s += [5] if not 3 <= t <= 6 else []
        out.append([int(x) for x in rng.permutation(s)])
    return out


SCHEDULE = _schedule()
N_FRAMES = 3 + max(sum(s in tick for tick in SCHEDULE) for s in range(N_SEQ))


@pytest.fixture(scope="module")
def scenes():
    """Six sequences, two per KITTI group, each rendered at its size through its calibration."""
    out = []
    for i in range(N_SEQ):
        K, (r, c) = KITTI[i // 2]
        s = synth.render_sequence("kitti", N_FRAMES, seed=500 + i, width=c, height=r, K=K)
        out.append((s["frames"], K, (r, c)))
    return out


def _copy(r):
    return {k: np.array(v) for k, v in r.items()}


def _assert_state(got, want, what=""):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), (what, k)
    assert got["status"] == want["status"], what


def _slot(images):
    out = np.zeros((len(images),) + SLOT, np.uint8)
    for k, im in enumerate(images):
        out[k, :im.shape[0], :im.shape[1]] = im
    return out


def _new_batch(scenes):
    return VOBatch(len(scenes), *SLOT, np.stack([K for _, K, _ in scenes]), OPT, frame_size=[sz for _, _, sz in scenes], **CAPS)


def _dev_out(n):
    import torch
    z = lambda *shape, dt=torch.int32: torch.zeros(shape, dtype=dt, device="cuda")
    return dict(status=z(n), n_inliers=z(n), n_lm=z(n), n_cand=z(n), pose_cw=z(n, 12, dt=torch.float64))


def _run(scenes, form, schedule=SCHEDULE, late=True, read_every_tick=True):
    """The schedule on one VOBatch of the six sequences.  A tick is a list of sequences (a listed step) or None (a full step).
    form: how the frames travel -- 'pageable', 'pinned', 'images', 'dev' (step_seqs_dev on device frames), 'sub1' / 'sub2'
    (host sets submitted one / two ticks ahead), 'subdev1' / 'subdev2' (device sets).  -> per tick (result rows, states)."""
    import torch
    vb = _new_batch(scenes)
    boot = [s for s in range(N_SEQ) if not (late and s == LATE)]
    vb.bootstrap([scenes[s][0][0] for s in boot], [scenes[s][0][2] for s in boot], seqs=boot)
    cnt = [0] * N_SEQ
    ticks = []   # (seqs or None, images in step order)
    for tick in schedule:
        seqs = list(range(N_SEQ)) if tick is None else tick
        ticks.append((tick, [scenes[s][0][3 + cnt[s]] for s in seqs]))
        for s in seqs:
            cnt[s] += 1
    ahead = int(form[-1]) if form.startswith("sub") else 0
    dev = form in ("dev", "subdev1", "subdev2")
    keep = []   # page-locked frames alive until the end of the run
    if dev:     # every device buffer exists before the first call: nothing in the run synchronises the device
        dframes = [torch.from_numpy(_slot(images)).cuda() for _, images in ticks]
        outs = [_dev_out(N_SEQ if tick is None else len(tick)) for tick, _ in ticks]
        torch.cuda.synchronize()

    def frames_of(t):
        tick, images = ticks[t]
        if form == "images":
            return images
        if dev:
            return dframes[t].data_ptr()
        arr = _slot(images)
        if form in ("pinned", "sub1", "sub2"):
            p = vb.pinned_empty(arr.shape, np.uint8)
            p[...] = arr
            keep.append(p)
            return p
        return arr

    def submit(t):
        tick = ticks[t][0]
        f = frames_of(t)
        if form.startswith("subdev"):
            vb.submit_frames_dev(f, seqs=tick)
        else:
            vb.submit_frames(f, seqs=tick)

    out, submitted = [], 0
    for t in range(len(ticks)):
        while ahead and submitted < min(t + ahead, len(ticks)):
            submit(submitted)
            submitted += 1
        if late and t == LATE_TICK:
            assert vb.bootstrap([scenes[LATE][0][0]], [scenes[LATE][0][2]], seqs=[LATE])["status"][0] == VOBatch.OK
        tick = ticks[t][0]
        if dev:
            o = outs[t]
            vb.step_dev(None if ahead else frames_of(t), {k: v.data_ptr() for k, v in o.items()}, seqs=tick)
            if read_every_tick:
                vb.ctx.sync()
                r = {k: v.cpu().numpy() for k, v in o.items()}
            else:
                r = None
        else:
            r = _copy(vb.step(None if ahead else frames_of(t), seqs=tick))
        out.append((r, [vb.read_state(s) for s in range(N_SEQ)] if read_every_tick else None))
    if not read_every_tick:
        vb.ctx.sync()
        out = [({k: v.cpu().numpy() for k, v in o.items()}, None) for o in outs]
        out[-1] = (out[-1][0], [vb.read_state(s) for s in range(N_SEQ)])
    vb.close()
    return out


@pytest.fixture(scope="module")
def ref_run(scenes):
    return _run(scenes, "pageable")


def _run_one(frames, K, size, n_steps):
    """a batch of one fed only its own frames with plain steps: states[0] before the bootstrap, states[1 + i] after i steps"""
    one = VOBatch(1, *SLOT, K, OPT, frame_size=[size], **CAPS)
    states = [one.read_state(0)]
    assert one.bootstrap([frames[0]], [frames[2]])["status"][0] == VOBatch.OK
    states.append(one.read_state(0))
    rows = []
    for f in range(3, 3 + n_steps):
        rows.append(_copy(one.step([frames[f]])))
        states.append(one.read_state(0))
    one.close()
    return rows, states


def test_schedule_equals_batches_of_one(scenes, ref_run):
    n_steps = [sum(s in tick for tick in SCHEDULE) for s in range(N_SEQ)]
    ones = [_run_one(scenes[s][0], scenes[s][1], scenes[s][2], n_steps[s]) for s in range(N_SEQ)]
    cnt = [0] * N_SEQ
    prev = None
    for t, (tick, (rows, states)) in enumerate(zip(SCHEDULE, ref_run)):
        assert rows["status"].shape == (len(tick),)
        for k, s in enumerate(tick):
            want = ones[s][0][cnt[s]]
            for key in RES_KEYS:
                assert np.array_equal(rows[key][k], want[key][0]), (t, s, key)
            cnt[s] += 1
        for s in range(N_SEQ):
            booted = not (s == LATE and t < LATE_TICK)
            _assert_state(states[s], ones[s][1][cnt[s] + 1 if booted else 0], (t, s))
            if prev is not None and s not in tick and not (s == LATE and t == LATE_TICK):
                _assert_state(states[s], prev[s], ("unlisted changed", t, s))
        prev = states
    # the comparison covers live steps
    assert sum(st["status"] == VOBatch.OK for st in ref_run[-1][1]) >= 4
    assert all(ref_run[-1][1][s]["status"] == VOBatch.OK for s in (0, LATE, 5))


def _assert_runs_equal(a, b):
    assert len(a) == len(b)
    for t, ((ra, sa), (rb, sb)) in enumerate(zip(a, b)):
        for k in RES_KEYS:
            assert np.array_equal(ra[k], rb[k]), (t, k)
        if sa is not None and sb is not None:
            for s, (x, y) in enumerate(zip(sa, sb)):
                _assert_state(x, y, (t, s))


@pytest.mark.parametrize("form", ["pinned", "images", "dev", "sub1", "sub2", "subdev1", "subdev2"])
def test_forms_are_identical(scenes, ref_run, form):
    _assert_runs_equal(_run(scenes, form), ref_run)


def test_fifo_mixes_full_and_listed_sets(scenes):
    """full and listed sets alternate in the FIFO (submitted two ahead) and are consumed in order"""
    sched = [None, [3, 0, 5], None, [2, 1], [4, 0, 5, 3], None, [5]]
    direct = _run(scenes, "pageable", sched, late=False)
    _assert_runs_equal(_run(scenes, "sub2", sched, late=False), direct)
    _assert_runs_equal(_run(scenes, "subdev1", sched, late=False), direct)


def test_in_flight_lists(scenes, ref_run):
    """listed steps and submitted listed sets enqueued back to back, with no host synchronisation between them, equal the
    same schedule synchronised after every call: every step and every queued set keeps its own list"""
    for form in ("dev", "subdev2"):
        got = _run(scenes, form, read_every_tick=False)
        _assert_runs_equal(got, ref_run)
        for s in range(N_SEQ):
            _assert_state(got[-1][1][s], ref_run[-1][1][s], s)


def test_full_list_equals_plain_step(scenes):
    a, b, c = _new_batch(scenes), _new_batch(scenes), _new_batch(scenes)
    for vb in (a, b, c):
        vb.bootstrap([f[0] for f, _, _ in scenes], [f[2] for f, _, _ in scenes])
    perm = [3, 5, 0, 2, 4, 1]
    for f in range(3, 7):
        images = [fr[f] for fr, _, _ in scenes]
        ra = _copy(a.step(images))
        rb = _copy(b.step(images, seqs=np.arange(N_SEQ)))
        rc = _copy(c.step([images[s] for s in perm], seqs=perm))
        for k in RES_KEYS:
            assert np.array_equal(ra[k], rb[k]), (f, k)
            assert np.array_equal(ra[k][perm], rc[k]), (f, k)
    for s in range(N_SEQ):
        _assert_state(b.read_state(s), a.read_state(s), s)
        _assert_state(c.read_state(s), a.read_state(s), s)
    for vb in (a, b, c):
        vb.close()


def test_listed_but_not_ok(scenes):
    """A never-loaded IDLE sequence and one driven to FEW_POINTS by blank frames report what the full step reports; both
    can then be bootstrapped and continue"""
    sc = scenes[:3]
    full, listed = _new_batch(sc), _new_batch(sc)
    for vb in (full, listed):
        vb.bootstrap([sc[s][0][0] for s in (0, 2)], [sc[s][0][2] for s in (0, 2)], seqs=[0, 2])
    blank = [np.zeros(sz, np.uint8) for _, _, sz in sc]
    for f in range(3, 5):
        images = [sc[0][0][f], blank[1], blank[2]]
        rf = _copy(full.step(images))
        rl = _copy(listed.step([blank[2], blank[1]], seqs=[2, 1]))
        for k in RES_KEYS:
            assert np.array_equal(rl[k], rf[k][[2, 1]]), (f, k)
    assert list(rl["status"]) == [VOBatch.FEW_POINTS, VOBatch.IDLE]
    assert not rl["n_inliers"].any() and not rl["pose_cw"].any()
    for s in (1, 2):
        _assert_state(listed.read_state(s), full.read_state(s), s)
    for vb in (full, listed):
        assert list(vb.bootstrap([sc[s][0][5] for s in (1, 2)], [sc[s][0][7] for s in (1, 2)], seqs=[1, 2])["status"]) == [VOBatch.OK] * 2
    for f in range(8, 11):
        rf = _copy(full.step([sc[s][0][f] for s in range(3)]))
        rl = _copy(listed.step([sc[s][0][f] for s in (2, 1)], seqs=[2, 1]))
        for k in RES_KEYS:
            assert np.array_equal(rl[k], rf[k][[2, 1]]), (f, k)
    assert list(rl["status"]) == [VOBatch.OK] * 2
    for s in (1, 2):
        _assert_state(listed.read_state(s), full.read_state(s), s)
    full.close()
    listed.close()


def test_refusals(scenes):
    import torch
    vb = _new_batch(scenes)
    vb.bootstrap([f[0] for f, _, _ in scenes], [f[2] for f, _, _ in scenes])
    lib, h = vb.ctx.lib, vb.h
    img = lambda s, f: scenes[s][0][f]
    before = [vb.read_state(s) for s in range(N_SEQ)]
    launches = vb.ctx.launch_count()
    res = {k: np.zeros((N_SEQ, 12) if k == "pose_cw" else N_SEQ, np.float64 if k == "pose_cw" else np.int32) for k in RES_KEYS}
    rp = [res[k].ctypes.data_as(C.POINTER(C.c_double) if k == "pose_cw" else c_i32p) for k in RES_KEYS]
    dev_out = _dev_out(N_SEQ)
    dp = [dev_out[k].data_ptr() for k in RES_KEYS]
    frames = _slot([img(0, 3), img(1, 3)])
    dframes = torch.from_numpy(frames).cuda()
    torch.cuda.synchronize()

    def seq_arr(seqs):
        a = np.ascontiguousarray(seqs, np.int32)
        return a, a.ctypes.data_as(c_i32p)

    def c_refusals(waiting_list=None):
        """every refusal of the four calls through the C ABI"""
        bad_lists = [(0, [0]), (N_SEQ + 1, list(range(N_SEQ)) + [0]), (2, [0, N_SEQ]), (2, [-1, 0]), (2, [1, 1])]
        fp = frames.ctypes.data_as(c_u8p)
        for n, seqs in bad_lists:
            a, p = seq_arr(seqs + [0] * max(0, n - len(seqs)))
            assert lib.b200vo_loop_step_seqs(h, n, p, fp, *rp) == -1, seqs
            assert lib.b200vo_loop_step_seqs_dev(h, n, p, dframes.data_ptr(), *dp) == -1, seqs
            assert lib.b200vo_loop_submit_frames_seqs(h, n, p, fp) == -1, seqs
            assert lib.b200vo_loop_submit_frames_seqs_dev(h, n, p, dframes.data_ptr()) == -1, seqs
        a, p = seq_arr([0, 1])
        assert lib.b200vo_loop_step_seqs(h, 2, None, fp, *rp) == -1
        assert lib.b200vo_loop_step_seqs(h, 2, p, fp, None, *rp[1:]) == -1
        assert lib.b200vo_loop_step_seqs_dev(h, 2, p, dframes.data_ptr(), dp[0], None, *dp[2:]) == -1
        assert lib.b200vo_loop_submit_frames_seqs(h, 2, p, None) == -1
        assert lib.b200vo_loop_submit_frames_seqs_dev(h, 2, None, dframes.data_ptr()) == -1
        if waiting_list is None:   # frames == NULL with nothing submitted
            assert lib.b200vo_loop_step_seqs(h, 2, p, None, *rp) == -1
            assert lib.b200vo_loop_step_seqs_dev(h, 2, p, None, *dp) == -1
        else:   # frames passed while a set waits; NULL with another list, or by the plain step
            assert lib.b200vo_loop_step_seqs(h, 2, p, fp, *rp) == -1
            assert lib.b200vo_loop_step_seqs_dev(h, 2, p, dframes.data_ptr(), *dp) == -1
            for other in ([1, 0], [0], [0, 1, 2]):
                a2, p2 = seq_arr(other)
                assert lib.b200vo_loop_step_seqs(h, len(other), p2, None, *rp) == -1, other
                assert lib.b200vo_loop_step_seqs_dev(h, len(other), p2, None, *dp) == -1, other
            assert lib.b200vo_loop_step(h, None, *rp) == -1
            assert lib.b200vo_loop_step_dev(h, None, *dp) == -1

    def py_refusals():
        for seqs in ([], [0, 0], [N_SEQ], [-1], [[0, 1]], [0.5], list(range(N_SEQ + 1))):
            with pytest.raises(ValueError):
                vb.step(frames[:max(len(seqs), 1)], seqs=seqs)
            with pytest.raises(ValueError):
                vb.step_dev(dframes.data_ptr(), {k: v.data_ptr() for k, v in dev_out.items()}, seqs=seqs)
            with pytest.raises(ValueError):
                vb.submit_frames(frames, seqs=seqs)
            with pytest.raises(ValueError):
                vb.submit_frames_dev(dframes.data_ptr(), seqs=seqs)
        for bad in (frames[:1], frames[:, :100], frames.astype(np.int16), [img(0, 3)], [img(0, 3), img(2, 3)]):   # sequence 1 is 376 x 1241, sequence 2's image 375 x 1242
            with pytest.raises(ValueError):
                vb.step(bad, seqs=[0, 1])
        with pytest.raises(ValueError):   # pageable frames cannot be submitted
            vb.submit_frames(frames, seqs=[0, 1])

    def unchanged():
        assert vb.ctx.launch_count() == launches
        for s in range(N_SEQ):
            _assert_state(vb.read_state(s), before[s], s)

    c_refusals()
    py_refusals()
    with pytest.raises(ValueError):
        vb.step(None, seqs=[0, 1])
    unchanged()
    # a waiting listed set: everything else is refused, and the matching call still consumes it
    pinned = vb.pinned_empty(frames.shape, np.uint8)
    pinned[...] = frames
    vb.submit_frames(pinned, seqs=[0, 1])
    c_refusals(waiting_list=[0, 1])
    py_refusals()
    with pytest.raises(ValueError):
        vb.step(None)
    with pytest.raises(ValueError):
        vb.step(None, seqs=[1, 0])
    unchanged()
    r = _copy(vb.step(None, seqs=[0, 1]))
    assert list(r["status"]) == [VOBatch.OK] * 2
    # a waiting full set is refused by the listed step and consumed by the plain one
    full = vb.pinned_frames()[0]
    full[...] = _slot([img(s, 4 if s < 2 else 3) for s in range(N_SEQ)])
    vb.submit_frames(full)
    before = [vb.read_state(s) for s in range(N_SEQ)]
    launches = vb.ctx.launch_count()
    for seqs in ([0, 1], list(range(N_SEQ))):
        with pytest.raises(ValueError):
            vb.step(None, seqs=seqs)
    unchanged()
    assert list(vb.step(None)["status"]) == [VOBatch.OK] * N_SEQ
    vb.close()
