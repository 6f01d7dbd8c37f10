"""bench.py contract pieces that can run without a GPU: the reference arm (cv2 on the host cores) prints ONE JSON
line with the keys the driver reads; the B200 arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    pytest.importorskip("cv2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-seqs", "2", "--batch", "2", "--frames", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_b200_arm_fails_loudly_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert "no CPU fallback" in (out.stderr + out.stdout)


# ---- the host loops of the B200 arm against a fake SequenceBatch: every (--steps, --warmup) the driver may pass ----
class _FakeCtx:
    def __init__(self):
        self.synced = 0

    def sync(self):
        self.synced += 1

    def last_gpu_ms(self):
        return 0.1


class _FakeBatch:
    """Stands in for batch.SequenceBatch: checks what the loops hand over, computes nothing."""
    instances = []

    def __init__(self, batch, rows, cols, K, **kw):
        import numpy as np
        self.batch, self.rows, self.cols = batch, rows, cols
        self.L, self.Cn = kw["max_landmarks"], kw["max_candidates"]
        self.queued, self.steps, self.closed = 0, 0, False
        self.np = np
        _FakeBatch.instances.append(self)

    def pinned_frames(self, n):
        return self.np.zeros((n, self.batch, self.rows, self.cols), self.np.uint8)

    def pinned_like(self, a):
        return a.copy()

    def pinned_empty(self, shape, dtype):
        return self.np.zeros(shape, dtype)

    def prime(self, frames):
        assert frames.shape[-2:] == (self.rows, self.cols)
        self.queued = 0

    def submit_frames(self, frames):
        assert frames.shape == (self.batch, self.rows, self.cols)
        assert self.queued < 2, "more than two frame sets waiting"
        self.queued += 1

    def step(self, frames, lm_pts, lm_obj, n_lm, cand_pts=None, n_cand=None):
        if frames is None:
            assert self.queued > 0, "frames=None without a submitted set"
            self.queued -= 1
        else:
            assert self.queued == 0
        assert lm_pts.shape == (self.batch, self.L, 2) and lm_obj.shape == (self.batch, self.L, 3) and n_lm.shape == (self.batch,)
        self.steps += 1
        return {}

    def close(self):
        self.closed = True


def _small_args(bench, steps, warmup):
    return bench.parse(["--steps", str(steps), "--warmup", str(warmup), "--batch", "2", "--frames", "3", "--landmarks", "40",
                        "--candidates", "30", "--distinct", "1", "--no-cpu-baseline"])


@pytest.fixture(scope="module")
def bench_mod():
    sys.path.insert(0, ROOT)
    import importlib
    return importlib.import_module("bench")


@pytest.mark.parametrize("steps", [1, 5, 20, 200])
@pytest.mark.parametrize("warmup", [0, 3, 5])
def test_single_sequence_extra_never_indexes_out_of_range(bench_mod, monkeypatch, steps, warmup):
    """Round 1's bench crashed with IndexError under --steps 20 --warmup 5 (a frame-order list sized for --steps 200)."""
    from monocular_visual_odometry_va4mr_b200 import batch, workload
    monkeypatch.setattr(batch, "SequenceBatch", _FakeBatch)
    args = _small_args(bench_mod, steps, warmup)
    opts = workload.REFERENCE_OPTIONS[args.shape]
    _FakeBatch.instances.clear()
    out = bench_mod.measure_single(args, opts, _FakeCtx(), max(warmup, 3))
    fb = _FakeBatch.instances[-1]
    n1 = bench_mod.single_plan(steps, max(warmup, 3))[0]
    assert fb.closed and fb.queued == 0 and fb.steps == max(warmup, 3) + n1 + 1
    assert out["frames"] == n1 and out["value"] > 0 and out["ms_per_frame_spread"]["n"] == n1


@pytest.mark.parametrize("steps", [1, 5, 20, 200])
@pytest.mark.parametrize("warmup", [0, 3, 5])
@pytest.mark.parametrize("prefetch", [False, True])
def test_host_loops_for_every_step_count(bench_mod, steps, warmup, prefetch):
    from monocular_visual_odometry_va4mr_b200 import workload
    args = _small_args(bench_mod, steps, warmup)
    opts = workload.REFERENCE_OPTIONS[args.shape]
    wl = bench_mod.make_workload(args, 2, 0) if not hasattr(test_host_loops_for_every_step_count, "wl") else test_host_loops_for_every_step_count.wl
    test_host_loops_for_every_step_count.wl = wl
    arm = object.__new__(bench_mod.Arm)
    arm.args, arm.opts, arm.ctx, arm.wl, arm.world, arm.local, arm.total = args, opts, _FakeCtx(), wl, 1, 0, 2
    arm.sb = _FakeBatch(wl.batch, wl.h, wl.w, wl.K, max_landmarks=wl.L, max_candidates=wl.Cn)
    arm.K, arm.W = max(steps, 1), max(warmup, 3)
    arm.barrier = lambda: None
    dt, wall, devms = arm.timed_host_loop(prefetch)
    assert dt > 0 and len(wall) == arm.K == len(devms)
    assert arm.sb.queued == 0 and arm.sb.steps == arm.K + arm.W + (1 if prefetch else 0)


def _fake_step_results(wl, seed):
    import numpy as np
    rng = np.random.default_rng(seed)
    b, L, Cn = wl.batch, wl.L, wl.Cn
    return {"lm_next": rng.random((b, L, 2), np.float32), "lm_status": rng.integers(0, 2, (b, L), np.uint8),
            "cand_next": rng.random((b, Cn, 2), np.float32), "cand_status": rng.integers(0, 2, (b, Cn), np.uint8),
            "pose": rng.random((b, 6)), "pnp_ok": np.ones(b, np.uint8), "inlier_mask": rng.integers(0, 2, (b, L), np.uint8),
            "n_inliers": rng.integers(0, L, b).astype(np.int32)}


def test_dump_outputs_writes_the_last_timed_step(bench_mod, tmp_path):
    import numpy as np
    args = _small_args(bench_mod, 4, 3)
    wl = bench_mod.make_workload(args, 2, 5)
    arm = object.__new__(bench_mod.Arm)
    arm.wl = wl
    last = _fake_step_results(wl, 0)
    t = 3 + 4 - 1
    bench_mod.dump_outputs(arm, {"timed_last": last, "timed_last_t": t}, str(tmp_path))
    f = arm.fo(t)
    got = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert sorted(got) == sorted(list(last) + ["sequence_index"])
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["pose"].dtype == np.float64 and np.array_equal(got["pose"], last["pose"])
    assert np.array_equal(got["sequence_index"], [5, 6]) and np.array_equal(got["n_inliers"], last["n_inliers"])
    for s in range(wl.batch):
        nl, nc = wl.n_lm[f, s], wl.n_cand[f, s]
        assert np.array_equal(got["lm_next"][s, :nl], last["lm_next"][s, :nl]) and not got["lm_next"][s, nl:].any()
        assert np.array_equal(got["lm_status"][s, :nl], last["lm_status"][s, :nl]) and not got["lm_status"][s, nl:].any()
        assert np.array_equal(got["inlier_mask"][s, :nl], last["inlier_mask"][s, :nl]) and not got["inlier_mask"][s, nl:].any()
        assert np.array_equal(got["cand_next"][s, :nc], last["cand_next"][s, :nc]) and not got["cand_next"][s, nc:].any()


def test_dump_outputs_samples_sequences_above_the_size_limit(bench_mod, tmp_path, monkeypatch):
    import numpy as np
    args = _small_args(bench_mod, 4, 3)
    wl = bench_mod.make_workload(args, 6, 0)
    arm = object.__new__(bench_mod.Arm)
    arm.wl = wl
    last = _fake_step_results(wl, 1)
    full = tmp_path / "full"
    bench_mod.dump_outputs(arm, {"timed_last": last, "timed_last_t": 7}, str(full))
    limit = sum(p.stat().st_size for p in full.glob("*.npy")) // 2
    monkeypatch.setattr(bench_mod, "DUMP_BYTES", limit)
    for run in ("a", "b"):
        bench_mod.dump_outputs(arm, {"timed_last": last, "timed_last_t": 7}, str(tmp_path / run))
        assert sum(p.stat().st_size for p in (tmp_path / run).glob("*.npy")) <= limit
    rows = np.load(tmp_path / "a" / "sequence_index.npy").astype(int)
    assert 0 < len(rows) < wl.batch and np.array_equal(rows, np.load(tmp_path / "b" / "sequence_index.npy"))
    for p in full.glob("*.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / p.name), np.load(p)[rows]), p.name


def test_frame_at_is_total_and_matches_frame_order():
    from monocular_visual_odometry_va4mr_b200 import workload
    for F in (1, 2, 3, 6):
        order = workload.frame_order(F, 50)
        assert len(order) == 51 and all(0 <= f < F for f in order)
        assert order == [workload.frame_at(F, t) for t in range(51)]
        assert all(abs(order[t + 1] - order[t]) <= 1 for t in range(50))   # always a small-baseline pair
        assert workload.frame_at(F, 10 ** 6) in range(F)


def test_extras_are_guarded(bench_mod):
    out = bench_mod.guarded(lambda: [][3])
    assert "IndexError" in out["error"]
    assert bench_mod.guarded(lambda: 5) == 5


def test_shard_plan_strong_and_weak(bench_mod):
    for world in (1, 2, 4, 8):
        blocks = [bench_mod.shard_plan(64, world, r, "strong") for r in range(world)]
        assert sum(b[1] for b in blocks) == 64 and all(b[2] == 64 for b in blocks)
        assert [b[0] for b in blocks] == [r * (64 // world) for r in range(world)]
        weak = [bench_mod.shard_plan(64, world, r, "weak") for r in range(world)]
        assert all(b[1] == 64 and b[2] == 64 * world for b in weak) and [b[0] for b in weak] == [64 * r for r in range(world)]


def test_workload_is_independent_of_the_sharding():
    import numpy as np
    from monocular_visual_odometry_va4mr_b200 import workload
    kw = dict(n_frames=2, n_landmarks=30, n_candidates=20, n_distinct=3, seed=0)
    full = workload.TrackWorkload("kitti", batch=6, first_index=0, **kw)
    part = workload.TrackWorkload("kitti", batch=2, first_index=4, **kw)
    for name in ("frames", "lm_pts", "lm_obj", "n_lm", "cand_pts", "n_cand"):
        assert np.array_equal(getattr(full, name)[:, 4:6], getattr(part, name)), name
