#!/usr/bin/env python
"""The device-resident loop with a camera per sequence (VOBatch with K of shape (batch, 3, 3)) against one shared camera and
against what per-camera batches cost.

  python benchmarks/bench_vo_intrinsics.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

The workload of bench_vo_loop.py: 64 KITTI-shaped sequences over 16 rendered scenes, visited forwards and backwards
(workload.frame_at), with the reference's KITTI options.  Scene d is rendered through its own camera: the KITTI calibration
d % 3 (sequences 00-02, 03, 04-12) with fx and fy scaled by up to 3 % and cx, cy moved by up to 4 pixels.  Sequence s shows
scene s % distinct.  Every sequence is bootstrapped on the device (VOBatch.bootstrap) on frames frame_at(F, k) and
frame_at(F, k + 2), k = s // distinct, then stepped with VOBatch.step_dev, frames resident on the device and submitted one
step ahead.  Three forms:

  (a) per_sequence_K  one VOBatch of all sequences, each with its scene's camera
  (b) shared_K        one VOBatch of all sequences with the KITTI 00-02 camera: the operating point of one calibration
  (c) per_camera      one VOBatch per distinct camera (16 batches of 4), stepped back to back: what one K per batch costs

Each run times `--steps` steps after `--warmup` steps (wall clock around work that ends in a device synchronise); the forms
alternate.  (a) and (c) must leave every sequence in the same state, array for array.  Prints one JSON line: ms per step of
all sequences for each form, whether (a) and (c) agree, and the device name, power limit and max SM clock.
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
KITTI = [(718.856, 607.1928, 185.2157), (721.5377, 609.5593, 172.854), (707.0912, 601.8873, 183.1104)]


def scene_cameras(n):
    rng = np.random.default_rng(7)
    Ks = []
    for d in range(n):
        f, cx, cy = KITTI[d % 3]
        sx, sy = 1 + rng.uniform(-0.03, 0.03, 2)
        dx, dy = rng.uniform(-4, 4, 2)
        Ks.append(np.array([[f * sx, 0.0, cx + dx], [0.0, f * sy, cy + dy], [0.0, 0.0, 1.0]]))
    return Ks


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
    Ks = scene_cameras(D)
    scenes = [synth.render_sequence("kitti", F, seed=d, K=Ks[d])["frames"] for d in range(D)]
    rows, cols = scenes[0].shape[1:]
    start = [s // D for s in range(B)]
    K_seq = np.stack([Ks[s % D] for s in range(B)])
    period = 2 * F - 2
    n_total = args.warmup + args.steps
    sets = np.stack([np.stack([scenes[s % D][workload.frame_at(F, start[s] + 3 + t)] for s in range(B)]) for t in range(period)])
    f0 = np.stack([scenes[s % D][workload.frame_at(F, start[s])] for s in range(B)])
    f1 = np.stack([scenes[s % D][workload.frame_at(F, start[s] + 2)] for s in range(B)])
    caps = dict(max_landmarks=4096, max_candidates=8192, max_frames=n_total + 8)
    groups = [np.arange(d, B, D) for d in range(D)]           # the sequences of camera d
    dev_sets = torch.from_numpy(sets).cuda()
    grp_sets = [torch.from_numpy(np.ascontiguousarray(sets[:, g])).cuda() for g in groups]

    def outs(n):
        return dict(status=torch.zeros(n, dtype=torch.int32, device="cuda"), n_inliers=torch.zeros(n, dtype=torch.int32, device="cuda"),
                    n_lm=torch.zeros(n, dtype=torch.int32, device="cuda"), n_cand=torch.zeros(n, dtype=torch.int32, device="cuda"),
                    pose_cw=torch.zeros((n, 12), dtype=torch.float64, device="cuda"))

    out_all = outs(B)
    out_grp = [outs(len(g)) for g in groups]
    ptr_all = {k: v.data_ptr() for k, v in out_all.items()}
    ptr_grp = [{k: v.data_ptr() for k, v in o.items()} for o in out_grp]
    torch.cuda.synchronize()

    def run(loops):
        """loops: [(VOBatch, device frame sets, result pointers)], stepped back to back."""
        for vb, fs, _ in loops:
            vb.submit_frames_dev(fs[0].data_ptr())
        t0 = None
        for t in range(n_total):
            if t == args.warmup:
                loops[0][0].ctx.sync()
                t0 = time.perf_counter()
            for vb, fs, ptr in loops:
                if t + 1 < n_total:
                    vb.submit_frames_dev(fs[(t + 1) % period].data_ptr())
                vb.step_dev(None, ptr)
        loops[0][0].ctx.sync()
        return time.perf_counter() - t0

    def one_batch(K):
        vb = VOBatch(B, rows, cols, K, OPT, **caps)
        r = vb.bootstrap(f0, f1)
        return [vb], [(vb, dev_sets, ptr_all)], int((r["status"] == VOBatch.OK).sum())

    def per_camera():
        vbs = []
        ok = 0
        for d, g in enumerate(groups):
            vb = VOBatch(len(g), rows, cols, Ks[d], OPT, **caps)
            ok += int((vb.bootstrap(f0[g], f1[g])["status"] == VOBatch.OK).sum())
            vbs.append(vb)
        return vbs, [(vb, grp_sets[d], ptr_grp[d]) for d, vb in enumerate(vbs)], ok

    def states(vbs):
        if len(vbs) == 1:
            return [vbs[0].read_state(s) for s in range(B)]
        st = [None] * B
        for d, g in enumerate(groups):
            for j, s in enumerate(g):
                st[s] = vbs[d].read_state(j)
        return st

    forms = {"per_sequence_K": lambda: one_batch(K_seq), "shared_K": lambda: one_batch(synth.K_KITTI.copy()),
             "per_camera": per_camera}
    res = {k: [] for k in forms}
    boot_ok, ends = {}, {}
    for _ in range(args.runs):
        for name, make in forms.items():
            vbs, loops, ok = make()
            res[name].append(1e3 * run(loops) / args.steps)
            boot_ok[name] = ok
            ends[name] = states(vbs)
            for vb in vbs:
                vb.close()
    agree = all(all(np.array_equal(a[k], c[k], equal_nan=True) for k in STATE_KEYS)
                for a, c in zip(ends["per_sequence_K"], ends["per_camera"]))
    line = dict(bench="vo_intrinsics", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup, shape=f"kitti {cols}x{rows}",
                ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                frames_per_s={k: round(B * 1e3 / min(vs), 1) for k, vs in res.items()},
                bootstrap_ok=boot_ok, final_status_ok={k: sum(int(x["status"] == VOBatch.OK) for x in v) for k, v in ends.items()},
                final_n_poses={k: sum(len(x["poses"]) for x in v) for k, v in ends.items()},
                per_sequence_K_equals_per_camera=bool(agree), **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    assert agree, "per-sequence K and per-camera batches leave different states"


if __name__ == "__main__":
    main()
