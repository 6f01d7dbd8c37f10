"""The batched device bootstrap (VOBatch.bootstrap, b200vo_loop_bootstrap): for every sequence it lists it must leave the
loop exactly as `load` of the host bootstrap chain (`initial_state(match_bootstrap_frames(...))`) leaves it, and touch no
other sequence."""
import numpy as np
import pytest

from mini_vo import REFERENCE_KITTI_OPTIONS as OPT
from monocular_visual_odometry_va4mr_b200 import synth
from monocular_visual_odometry_va4mr_b200.batch import VOBatch, initial_state, match_bootstrap_frames

pytestmark = pytest.mark.gpu

CAPS = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")
ROWS, COLS = 376, 1241


@pytest.fixture(scope="module")
def scenes():
    """The six KITTI-shaped sequences of test_vo_loop_gpu.py, with the host chain's bootstrap on frames 0 and 2."""
    out = []
    for seed in range(6):
        s = synth.render_sequence("kitti", 15, seed=100 + seed)
        st = initial_state(s["K"], OPT, *match_bootstrap_frames(s["frames"][0], s["frames"][2], OPT["feature_ratio"]))
        out.append((s["frames"], st))
    return s["K"], out


def _assert_state(got, want):
    for k in STATE_KEYS:
        assert got[k].shape == np.asarray(want[k]).shape and np.array_equal(got[k], want[k], equal_nan=True), k


def _copy(r):
    return {k: np.array(v) for k, v in r.items()}


def _step(vb, seqs, f):
    return _copy(vb.step(np.stack([fr[f] for fr, _ in seqs])))


def test_bootstrap_equals_host_chain(scenes):
    K, seqs = scenes
    dev = VOBatch(len(seqs), ROWS, COLS, K, OPT, **CAPS)
    host = VOBatch(len(seqs), ROWS, COLS, K, OPT, **CAPS)
    r = dev.bootstrap(np.stack([fr[0] for fr, _ in seqs]), np.stack([fr[2] for fr, _ in seqs]))
    assert list(r["status"]) == [VOBatch.OK] * len(seqs)
    for s, (fr, st) in enumerate(seqs):
        host.load(s, fr[2], st)
        assert r["num_pts"][s] == st["num_pts"]
        assert r["n_lm"][s] == len(st["lm"]) and r["n_cand"][s] == len(st["keys"])
        got = dev.read_state(s)
        assert got["status"] == VOBatch.OK
        _assert_state(got, host.read_state(s))
    for f in range(3, 6):
        rd, rh = _step(dev, seqs, f), _step(host, seqs, f)
        for k in rd:
            assert np.array_equal(rd[k], rh[k]), (f, k)


def test_subset_isolation_and_revival(scenes):
    K, seqs = scenes
    _, sa = seqs[2]
    few = dict(sa, lm=sa["lm"][:7], lm_kp=sa["lm_kp"][:7])
    vbs = [VOBatch(len(seqs), ROWS, COLS, K, OPT, **CAPS) for _ in range(2)]   # the second one never gets the call
    for vb in vbs:
        for s, (fr, st) in enumerate(seqs):
            vb.load(s, fr[2], few if s == 2 else st)
        r = _step(vb, seqs, 3)
        assert r["status"][2] == VOBatch.FEW_POINTS
    vb, ctl = vbs
    (f2, _), (f4, st4) = seqs[2], seqs[4]
    r = vb.bootstrap(np.stack([f4[3], f2[3]]), np.stack([f4[4], f2[4]]), seqs=[4, 2])   # reverse index order
    assert list(r["status"]) == [VOBatch.OK, VOBatch.OK]
    for k, (fr, s) in enumerate([(f4, 4), (f2, 2)]):
        st = initial_state(K, OPT, *match_bootstrap_frames(fr[3], fr[4], OPT["feature_ratio"]))
        assert r["num_pts"][k] == st["num_pts"]
        _assert_state(vb.read_state(s), dict(st, poses=st["poses"]))
    others = [0, 1, 3, 5]
    for s in others:
        _assert_state(vb.read_state(s), ctl.read_state(s))
    rv, rc = _step(vb, seqs, 5), _step(ctl, seqs, 5)
    assert rv["status"][2] == VOBatch.OK and rv["n_inliers"][2] > 0    # the stopped sequence runs again
    assert rc["status"][2] == VOBatch.FEW_POINTS
    for k in rv:
        assert np.array_equal(rv[k][others], rc[k][others]), k
    for s in others:
        _assert_state(vb.read_state(s), ctl.read_state(s))


def test_failure_codes(scenes):
    K, seqs = scenes
    fr, st = seqs[0]
    vb = VOBatch(2, ROWS, COLS, K, OPT, **CAPS)
    vb.load(0, fr[2], st)
    vb.load(1, fr[2], st)
    before = vb.read_state(0)
    grey = np.full((1, ROWS, COLS), 128, np.uint8)
    r = vb.bootstrap(grey, grey, seqs=[0])
    assert r["status"][0] == VOBatch.NO_BOOTSTRAP and r["num_pts"][0] == 0
    after = vb.read_state(0)
    assert after["status"] == VOBatch.NO_BOOTSTRAP
    _assert_state(after, before)
    for f in (3, 4):
        r = vb.step(np.stack([fr[f], fr[f]]))
        assert r["status"][0] == VOBatch.NO_BOOTSTRAP and r["n_inliers"][0] == 0 and r["status"][1] == VOBatch.OK
    _assert_state(vb.read_state(0), before)

    small = VOBatch(1, ROWS, COLS, K, OPT, **dict(CAPS, max_landmarks=len(st["lm"]) - 1))
    small.load(0, fr[2], dict(st, lm=st["lm"][:5], lm_kp=st["lm_kp"][:5]))
    before = small.read_state(0)
    r = small.bootstrap(fr[None, 0], fr[None, 2])
    assert r["status"][0] == VOBatch.OVERFLOW and r["num_pts"][0] == st["num_pts"]
    after = small.read_state(0)
    assert after["status"] == VOBatch.OVERFLOW
    _assert_state(after, before)


def test_validation(scenes):
    K, seqs = scenes
    vb = VOBatch(3, ROWS, COLS, K, OPT, **CAPS)
    for s in range(3):
        fr, st = seqs[s]
        vb.load(s, fr[2], st)
    before = [vb.read_state(s) for s in range(3)]
    f = np.stack([seqs[0][0][0]] * 2)
    n0 = vb.ctx.launch_count()
    bad = [dict(frames0=f, frames1=f, seqs=[0, 3]), dict(frames0=f, frames1=f, seqs=[1, 1]),
           dict(frames0=f[:, :-1], frames1=f[:, :-1], seqs=[0, 1]), dict(frames0=f[:0], frames1=f[:0], seqs=[])]
    for kw in bad:
        with pytest.raises(ValueError):
            vb.bootstrap(**kw)
    assert vb.ctx.launch_count() == n0
    for s in range(3):
        now = vb.read_state(s)
        assert now["status"] == before[s]["status"]
        _assert_state(now, before[s])


def test_batching_is_real(scenes):
    K, seqs = scenes
    vb = VOBatch(len(seqs), ROWS, COLS, K, OPT, **CAPS)
    f0, f1 = np.stack([fr[0] for fr, _ in seqs]), np.stack([fr[2] for fr, _ in seqs])
    vb.bootstrap(f0, f1)                                      # warm: workspaces sized
    n0 = vb.ctx.launch_count()
    vb.bootstrap(f0[:1], f1[:1], seqs=[0])
    one = vb.ctx.launch_count() - n0
    n0 = vb.ctx.launch_count()
    vb.bootstrap(f0, f1)
    six = vb.ctx.launch_count() - n0
    assert six < 1.5 * one, (one, six)


def test_frames_beyond_one_sift_chunk():
    """14 sequences = 28 frames: more than one chunk of KITTI-shaped scale spaces fits the SIFT workspace budget, so the
    keypoint rows of later chunks follow those of earlier ones."""
    scenes = [synth.render_sequence("kitti", 3, seed=200 + s) for s in range(14)]
    K = scenes[0]["K"]
    f0 = np.stack([s["frames"][0] for s in scenes])
    f1 = np.stack([s["frames"][2] for s in scenes])
    dev = VOBatch(len(scenes), ROWS, COLS, K, OPT, **CAPS)
    host = VOBatch(len(scenes), ROWS, COLS, K, OPT, **CAPS)
    r = dev.bootstrap(f0, f1)
    for s in range(len(scenes)):
        try:
            st = initial_state(K, OPT, *match_bootstrap_frames(f0[s], f1[s], OPT["feature_ratio"]))
        except ValueError:
            assert r["status"][s] == VOBatch.NO_BOOTSTRAP
            continue
        assert r["status"][s] == VOBatch.OK and r["num_pts"][s] == st["num_pts"]
        host.load(s, f1[s], st)
        _assert_state(dev.read_state(s), host.read_state(s))
    assert (r["status"] == VOBatch.OK).sum() >= 12
