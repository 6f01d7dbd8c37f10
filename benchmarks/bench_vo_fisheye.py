#!/usr/bin/env python
"""The device-resident loop with per-sequence fisheye lenses (VOBatch.set_distortion(model="fisheye")) next to the same loop
with pinhole lenses and without lenses, plus the time to build the maps of a whole batch.

  python benchmarks/bench_vo_fisheye.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

The workload of bench_vo_distortion.py: 64 KITTI-shaped sequences (1241 x 376) over 16 rendered scenes, bootstrapped on the
device and stepped with VOBatch.step_dev, frames resident on the device and submitted one step ahead.  Three forms, set
before the bootstrap:

  (a) none        no sequence has a lens: the pyramid builder copies the frames
  (b) pinhole     every sequence has a mild KITTI-like 5-coefficient pinhole lens, raw camera = K
  (c) fisheye     every sequence has a fisheye lens whose raw camera has 0.8 x K's focal length, undistorted into K

Level 0 of (b) and (c) is gathered through a map of the same layout, so their step times should match; the maps differ
only in how they are evaluated.  The rendered frames are treated as raw camera output, so the point counts of the three
forms differ; the line reports the final landmark counts.  Each run times `--steps` steps after `--warmup` steps (wall
clock around work that ends in a device synchronise); the forms alternate.  The map build is timed as the wall clock of a
synchronous set_distortion of all sequences (the settings upload, the map kernel and its synchronise), best of `--reps`, for
both models.  Prints one JSON line with the device name, power limit and max SM clock.
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

PINHOLE = [-0.06, 0.01, 0.0004, -0.0003, 0.0]
FISHEYE = [0.02, 0.01, -0.003, 0.0002]
RAW_F = 0.8


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--steps", type=int, default=150)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    from monocular_visual_odometry_va4mr_b200 import synth, workload
    from monocular_visual_odometry_va4mr_b200.batch import VOBatch

    B, D, F = args.batch, args.distinct, args.frames
    seqs0 = [synth.render_sequence("kitti", F, seed=d) for d in range(D)]
    K = seqs0[0]["K"]
    K_raw = K.copy()
    K_raw[0, 0] *= RAW_F
    K_raw[1, 1] *= RAW_F
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
    every = np.arange(B)
    lens = {"none": None,
            "pinhole": (np.tile(PINHOLE, (B, 1)), "pinhole", None),
            "fisheye": (np.tile(FISHEYE, (B, 1)), "fisheye", np.tile(K_raw, (B, 1, 1)))}

    def run(form):
        """-> (ms per step, bootstraps OK, final states)"""
        vb = VOBatch(B, rows, cols, K, OPT, **caps)
        if lens[form]:
            vb.set_distortion(every, *lens[form])
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

    def map_build_ms():
        """best wall clock of a synchronous set_distortion of every sequence, per model"""
        vb = VOBatch(B, rows, cols, K, OPT, **caps)
        res = {}
        for form in ("pinhole", "fisheye"):
            vb.set_distortion(every, *lens[form])   # the map memory is allocated with the first lens
            best = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                vb.set_distortion(every, *lens[form])
                best.append(1e3 * (time.perf_counter() - t0))
            res[form] = round(min(best), 4)
        vb.close()
        return res

    res = {k: [] for k in lens}
    boot_ok, ends = {}, {}
    for _ in range(args.runs):
        for form in lens:
            ms, ok, states = run(form)
            res[form].append(ms)
            boot_ok[form], ends[form] = ok, states
    line = dict(bench="vo_fisheye", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup, shape=f"{cols}x{rows}",
                pinhole=PINHOLE, fisheye=FISHEYE, fisheye_raw_focal_scale=RAW_F,
                ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                frames_per_s={k: round(B * 1e3 / min(vs), 1) for k, vs in res.items()},
                bootstrap_ok=boot_ok, final_status_ok={k: sum(int(x["status"] == VOBatch.OK) for x in v) for k, v in ends.items()},
                final_landmarks={k: sum(len(x["lm"]) for x in v) for k, v in ends.items()},
                map_build_ms_all_sequences=map_build_ms(), **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
