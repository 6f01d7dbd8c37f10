#!/usr/bin/env python
"""The device-resident loop with a frame size per sequence (VOBatch with frame_size) against what per-size batches cost.

  python benchmarks/bench_vo_frame_size.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

The workload of bench_vo_loop.py at KITTI's three native image sizes: 64 sequences over 16 rendered scenes, visited forwards
and backwards (workload.frame_at), with the reference's KITTI options.  Scene d belongs to KITTI group d % 3 (sequences
00-02: 1241 x 376, 03: 1242 x 375, 04-12: 1226 x 370) and is rendered at that group's size through its calibration.  Sequence
s shows scene s % distinct.  Every sequence is bootstrapped on the device (VOBatch.bootstrap) on frames frame_at(F, k) and
frame_at(F, k + 2), k = s // distinct, then stepped with VOBatch.step_dev, frames resident on the device and submitted one
step ahead.  Two forms:

  (a) per_sequence_size  one VOBatch of all sequences in 1242 x 376 slots, each with its own frame size
  (b) per_size           one VOBatch per frame size (three batches), stepped back to back: what one size per batch costs

Each run times `--steps` steps after `--warmup` steps (wall clock around work that ends in a device synchronise); the forms
alternate.  Both must leave every sequence in the same state, array for array.  Prints one JSON line: ms per step of all
sequences for each form, whether they agree, and the device name, power limit and max SM clock.
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
# KITTI groups 00-02, 03, 04-12: fx = fy, cx, cy and the image size (rows, cols)
KITTI = [(718.856, 607.1928, 185.2157, (376, 1241)), (721.5377, 609.5593, 172.854, (375, 1242)),
         (707.0912, 601.8873, 183.1104, (370, 1226))]
SLOT = (376, 1242)


def group_camera(g):
    f, cx, cy, _ = KITTI[g]
    return np.array([[f, 0.0, cx], [0.0, f, cy], [0.0, 0.0, 1.0]])


def slot_layout(images):
    out = np.zeros((len(images),) + SLOT, np.uint8)
    for k, im in enumerate(images):
        out[k, :im.shape[0], :im.shape[1]] = im
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
    grp = [s % D % 3 for s in range(B)]                       # the KITTI group of sequence s
    scenes = [synth.render_sequence("kitti", F, seed=d, width=KITTI[d % 3][3][1], height=KITTI[d % 3][3][0],
                                    K=group_camera(d % 3))["frames"] for d in range(D)]
    start = [s // D for s in range(B)]
    K_seq = np.stack([group_camera(g) for g in grp])
    sizes = np.int32([KITTI[g][3] for g in grp])
    period = 2 * F - 2
    n_total = args.warmup + args.steps
    img = lambda s, i: scenes[s % D][workload.frame_at(F, start[s] + i)]
    groups = [np.flatnonzero(np.int32(grp) == g) for g in range(3)]   # the sequences of size g
    caps = dict(max_landmarks=4096, max_candidates=8192, max_frames=n_total + 8)
    dev_sets = torch.from_numpy(np.stack([slot_layout([img(s, 3 + t) for s in range(B)]) for t in range(period)])).cuda()
    grp_sets = [torch.from_numpy(np.stack([np.stack([img(s, 3 + t) for s in g]) for t in range(period)])).cuda() for g in groups]

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

    def per_sequence_size():
        vb = VOBatch(B, *SLOT, K_seq, OPT, frame_size=sizes, **caps)
        r = vb.bootstrap([img(s, 0) for s in range(B)], [img(s, 2) for s in range(B)])
        return [vb], [(vb, dev_sets, ptr_all)], int((r["status"] == VOBatch.OK).sum())

    def per_size():
        vbs = []
        ok = 0
        for g, members in enumerate(groups):
            vb = VOBatch(len(members), *KITTI[g][3], group_camera(g), OPT, **caps)
            r = vb.bootstrap(np.stack([img(s, 0) for s in members]), np.stack([img(s, 2) for s in members]))
            ok += int((r["status"] == VOBatch.OK).sum())
            vbs.append(vb)
        return vbs, [(vb, grp_sets[g], ptr_grp[g]) for g, vb in enumerate(vbs)], ok

    def states(vbs):
        if len(vbs) == 1:
            return [vbs[0].read_state(s) for s in range(B)]
        st = [None] * B
        for g, members in enumerate(groups):
            for j, s in enumerate(members):
                st[s] = vbs[g].read_state(j)
        return st

    forms = {"per_sequence_size": per_sequence_size, "per_size": per_size}
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
                for a, c in zip(ends["per_sequence_size"], ends["per_size"]))
    line = dict(bench="vo_frame_size", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup,
                shapes={f"{c}x{r}": len(g) for (_, _, _, (r, c)), g in zip(KITTI, groups)}, slot=f"{SLOT[1]}x{SLOT[0]}",
                ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                frames_per_s={k: round(B * 1e3 / min(vs), 1) for k, vs in res.items()},
                bootstrap_ok=boot_ok, final_status_ok={k: sum(int(x["status"] == VOBatch.OK) for x in v) for k, v in ends.items()},
                final_n_poses={k: sum(len(x["poses"]) for x in v) for k, v in ends.items()},
                per_sequence_size_equals_per_size=bool(agree), **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    assert agree, "per-sequence sizes and per-size batches leave different states"


if __name__ == "__main__":
    main()
