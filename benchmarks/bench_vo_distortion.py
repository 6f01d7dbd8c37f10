#!/usr/bin/env python
"""The device-resident loop with per-sequence lens distortion (VOBatch.set_distortion) against the same loop without, and
the one-call b200vo_undistort against cv2.undistort on the host's cores.

  python benchmarks/bench_vo_distortion.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

The workload of bench_vo_masks.py: 64 KITTI-shaped sequences (1241 x 376) over 16 rendered scenes, bootstrapped on the
device and stepped with VOBatch.step_dev, frames resident on the device and submitted one step ahead.  Three forms, set
before the bootstrap:

  (a) none        no sequence has distortion: the pyramid builder copies the frames (the path of every batch before)
  (b) dist_all    every sequence has a mild KITTI-like 5-coefficient distortion: level 0 is gathered through its map
  (c) dist_half   the even sequences have it, the odd ones do not

The rendered frames are treated as raw camera output, so a distorted sequence tracks a (mildly) different image and its
point counts differ from the undistorted run's; the line reports the final landmark and candidate counts.  An undistorted
sequence of dist_half must end exactly as in none.  Each run times `--steps` steps after `--warmup` steps (wall clock around
work that ends in a device synchronise); the forms alternate.  The per-call part times cv2_compat.undistort (upload, map,
remap, download; host clock) and cv2.undistort with one thread and with every core of the host, on one 1241 x 376 frame.
Prints one JSON line with the device name, power limit and max SM clock.
"""

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "benchmarks"))

from bench_vo_loop import device_info  # noqa: E402
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT  # noqa: E402

STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses", "status")
DIST = [-0.06, 0.01, 0.0004, -0.0003, 0.0, 0.0, 0.0, 0.0]


def per_call(frame, K, reps=200):
    """ms per call of cv2_compat.undistort and of cv2.undistort (1 thread, all threads), best of three batches of reps"""
    from monocular_visual_odometry_va4mr_b200 import cv2_compat
    d = np.asarray(DIST[:5])
    out = {}

    def best(fn):
        fn()
        r = []
        for _ in range(3):
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            r.append(1e3 * (time.perf_counter() - t0) / reps)
        return round(min(r), 4)
    out["b200vo_undistort_ms"] = best(lambda: cv2_compat.undistort(frame, K, d))
    try:
        import cv2
    except ImportError:
        return out
    same = bool(np.array_equal(cv2_compat.undistort(frame, K, d), cv2.undistort(frame, K, d)))
    n = cv2.getNumThreads()
    cv2.setNumThreads(1)
    out["cv2_undistort_1_thread_ms"] = best(lambda: cv2.undistort(frame, K, d))
    cv2.setNumThreads(os.cpu_count() or n)
    out["cv2_undistort_all_threads_ms"] = best(lambda: cv2.undistort(frame, K, d))
    out["host_cpus"] = os.cpu_count()
    cv2.setNumThreads(n)
    out["equal_to_cv2"] = same
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    from monocular_visual_odometry_va4mr_b200 import synth, workload
    from monocular_visual_odometry_va4mr_b200.batch import VOBatch

    B, D, F = args.batch, args.distinct, args.frames
    seqs0 = [synth.render_sequence("kitti", F, seed=d) for d in range(D)]
    K = seqs0[0]["K"]
    scenes = [s["frames"] for s in seqs0]
    rows, cols = scenes[0][0].shape
    start = [s // D for s in range(B)]
    period = 2 * F - 2
    n_total = args.warmup + args.steps
    img = lambda s, i: scenes[s % D][workload.frame_at(F, start[s] + i)]
    caps = dict(max_landmarks=4096, max_candidates=8192, max_frames=n_total + 8)
    dev_sets = torch.from_numpy(np.stack([np.stack([img(s, 3 + t) for s in range(B)]) for t in range(period)])).cuda()
    out = dict(status=torch.zeros(B, dtype=torch.int32, device="cuda"), n_inliers=torch.zeros(B, dtype=torch.int32, device="cuda"),
               n_lm=torch.zeros(B, dtype=torch.int32, device="cuda"), n_cand=torch.zeros(B, dtype=torch.int32, device="cuda"),
               pose_cw=torch.zeros((B, 12), dtype=torch.float64, device="cuda"))
    ptr = {k: v.data_ptr() for k, v in out.items()}
    torch.cuda.synchronize()
    forms = {"none": [], "dist_all": list(range(B)), "dist_half": list(range(0, B, 2))}

    def run(distorted):
        """-> (ms per step, bootstraps OK, final states)"""
        vb = VOBatch(B, rows, cols, K, OPT, **caps)
        if distorted:
            vb.set_distortion(distorted, np.tile(DIST, (len(distorted), 1)))
        boot = vb.bootstrap(np.stack([img(s, 0) for s in range(B)]), np.stack([img(s, 2) for s in range(B)]))
        vb.submit_frames_dev(dev_sets[0].data_ptr())
        t0 = None
        for t in range(n_total):
            if t == args.warmup:
                vb.ctx.sync()
                t0 = time.perf_counter()
            if t + 1 < n_total:
                vb.submit_frames_dev(dev_sets[(t + 1) % period].data_ptr())
            vb.step_dev(None, ptr)
        vb.ctx.sync()
        ms = 1e3 * (time.perf_counter() - t0) / args.steps
        states = [vb.read_state(s) for s in range(B)]
        vb.close()
        return ms, int((boot["status"] == VOBatch.OK).sum()), states

    res = {k: [] for k in forms}
    boot_ok, ends = {}, {}
    for _ in range(args.runs):
        for name, distorted in forms.items():
            ms, ok, states = run(distorted)
            res[name].append(ms)
            boot_ok[name], ends[name] = ok, states
    plain = [s for s in range(B) if s not in forms["dist_half"]]
    agree = all(all(np.array_equal(ends["dist_half"][s][k], ends["none"][s][k], equal_nan=True) for k in STATE_KEYS) for s in plain)
    line = dict(bench="vo_distortion", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup, shape=f"{cols}x{rows}",
                dist=DIST, ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                frames_per_s={k: round(B * 1e3 / min(vs), 1) for k, vs in res.items()},
                bootstrap_ok=boot_ok, final_status_ok={k: sum(int(x["status"] == VOBatch.OK) for x in v) for k, v in ends.items()},
                final_landmarks={k: sum(len(x["lm"]) for x in v) for k, v in ends.items()},
                final_candidates={k: sum(len(x["keys"]) for x in v) for k, v in ends.items()},
                dist_half_undistorted_equal_none=bool(agree), per_call=per_call(scenes[0][0], K), **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    assert agree, "an undistorted sequence of dist_half ended differently from none"


if __name__ == "__main__":
    main()
