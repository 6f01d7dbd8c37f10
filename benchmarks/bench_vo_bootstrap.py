#!/usr/bin/env python
"""The batched device bootstrap (VOBatch.bootstrap) against the host bootstrap chain plus load.

  python benchmarks/bench_vo_bootstrap.py [--batch 64] [--distinct 16] [--frames 10] [--warmup 1] [--runs 3] [--out FILE]

The workload of bench_vo_loop.py: 64 KITTI-shaped sequences over 16 rendered scenes (workload.frame_at), with the
reference's KITTI options.  Sequence s uses scene s % distinct and bootstraps on frames frame_at(F, k) and
frame_at(F, k + 2), k = s // distinct.  Two forms leave the same loop state:

  (a) device  one VOBatch.bootstrap call for every sequence
  (b) host    per sequence: initial_state(K, options, *match_bootstrap_frames(f0, f1, ratio)) and VOBatch.load

Each run times one bootstrap of every sequence (wall clock around work that ends in a device synchronise); the forms
alternate, `--warmup` untimed runs first.  Both forms' states are compared array for array.  Prints one JSON line: ms per
bootstrap of all sequences for each form, whether the states agree, and the device name, power limit and max SM clock.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--distinct", type=int, default=16)
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    args = ap.parse_args()
    import torch
    from monocular_visual_odometry_va4mr_b200 import synth, workload
    from monocular_visual_odometry_va4mr_b200.batch import VOBatch, initial_state, match_bootstrap_frames

    B, D, F = args.batch, args.distinct, args.frames
    scenes = [synth.render_sequence("kitti", F, seed=d)["frames"] for d in range(D)]
    K = synth.SHAPES["kitti"][0].copy()
    rows, cols = scenes[0].shape[1:]
    f0 = np.stack([scenes[s % D][workload.frame_at(F, s // D)] for s in range(B)])
    f1 = np.stack([scenes[s % D][workload.frame_at(F, s // D + 2)] for s in range(B)])
    caps = dict(max_landmarks=4096, max_candidates=8192, max_frames=64)
    vb_dev = VOBatch(B, rows, cols, K, OPT, **caps)
    vb_host = VOBatch(B, rows, cols, K, OPT, **caps)

    def run_dev():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = vb_dev.bootstrap(f0, f1)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    def run_host():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(B):
            vb_host.load(s, f1[s], initial_state(K, OPT, *match_bootstrap_frames(f0[s], f1[s], OPT["feature_ratio"])))
        torch.cuda.synchronize()
        return time.perf_counter() - t0, None

    for _ in range(args.warmup):
        run_dev()
        run_host()
    res = {"device": [], "host": []}
    for _ in range(args.runs):
        res["device"].append(1e3 * run_dev()[0])
        res["host"].append(1e3 * run_host()[0])
    r = vb_dev.bootstrap(f0, f1)
    agree = True
    for s in range(B):
        a, b = vb_dev.read_state(s), vb_host.read_state(s)
        agree = agree and all(np.array_equal(a[k], b[k], equal_nan=True) for k in STATE_KEYS)
    line = dict(bench="vo_bootstrap", batch=B, distinct=D, frames=F, runs=args.runs, shape=f"kitti {cols}x{rows}",
                ms_per_bootstrap_of_all={k: [round(v, 2) for v in vs] for k, vs in res.items()},
                status_ok=int((r["status"] == VOBatch.OK).sum()), states_agree=bool(agree), **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    assert agree, "the two forms leave different states"


if __name__ == "__main__":
    main()
