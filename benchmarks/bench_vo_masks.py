#!/usr/bin/env python
"""The device-resident loop with per-sequence detection masks (VOBatch.set_detection_mask) against the same loop without.

  python benchmarks/bench_vo_masks.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

The workload of bench_vo_loop.py: 64 KITTI-shaped sequences (1241 x 376) over 16 rendered scenes, visited forwards and
backwards (workload.frame_at), with the reference's KITTI options.  Every sequence is bootstrapped on the device on frames
frame_at(F, k) and frame_at(F, k + 2), k = s // distinct, then stepped with VOBatch.step_dev, frames resident on the device
and submitted one step ahead.  Three forms, set before the bootstrap:

  (a) no_mask     no sequence has a mask: the detector runs without mask reads (the path of every batch before masks)
  (b) hood_all    every sequence masks a dash camera's hood (the bottom fifth of the frame, rounded shoulders)
  (c) hood_half   the even sequences mask the hood, the odd ones have no mask

Each run times `--steps` steps after `--warmup` steps (wall clock around work that ends in a device synchronise); the forms
alternate.  A masked sequence detects different corners, so its landmarks and candidates, and with them the tracking and
triangulation work of later steps, differ from the unmasked run's.  One untimed pass per form sums, over every step, the
landmarks and candidates each sequence holds after it (the points the next step tracks, and the candidates the
triangulation tests) and its PnP inliers, on the library's stream; the line reports them per step and sequence, with the
sequences still OK at the end.  An unmasked sequence of hood_half must end exactly as in no_mask.  Prints one JSON line
with the device name, power limit and max SM clock.
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
from mask_reference import hood_mask  # noqa: E402
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT  # noqa: E402

STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses", "status")


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
    hood = hood_mask((rows, cols))
    out = dict(status=torch.zeros(B, dtype=torch.int32, device="cuda"), n_inliers=torch.zeros(B, dtype=torch.int32, device="cuda"),
               n_lm=torch.zeros(B, dtype=torch.int32, device="cuda"), n_cand=torch.zeros(B, dtype=torch.int32, device="cuda"),
               pose_cw=torch.zeros((B, 12), dtype=torch.float64, device="cuda"))
    ptr = {k: v.data_ptr() for k, v in out.items()}
    torch.cuda.synchronize()
    forms = {"no_mask": [], "hood_all": list(range(B)), "hood_half": list(range(0, B, 2))}

    def run(masked, count=False):
        """-> (ms per step, bootstraps OK, final states, per-step sums of n_lm, n_cand, n_inliers over all sequences or None)"""
        vb = VOBatch(B, rows, cols, K, OPT, **caps)
        lib_stream = torch.cuda.ExternalStream(vb.ctx.stream())
        acc = torch.zeros(3, dtype=torch.int64, device="cuda")
        if masked:
            vb.set_detection_mask(masked, np.broadcast_to(hood, (len(masked), rows, cols)))
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
            if count and t >= args.warmup:     # ordered after the step on its stream; the timing of this pass is not used
                with torch.cuda.stream(lib_stream):
                    acc += torch.stack([out["n_lm"].sum(), out["n_cand"].sum(), out["n_inliers"].sum()])
        vb.ctx.sync()
        ms = 1e3 * (time.perf_counter() - t0) / args.steps
        states = [vb.read_state(s) for s in range(B)]
        work = (acc.cpu().numpy() / (args.steps * B)).round(1).tolist() if count else None
        vb.close()
        return ms, int((boot["status"] == VOBatch.OK).sum()), states, work

    res = {k: [] for k in forms}
    boot_ok, ends, work = {}, {}, {}
    for _ in range(args.runs):
        for name, masked in forms.items():
            ms, ok, states, _ = run(masked)
            res[name].append(ms)
            boot_ok[name], ends[name] = ok, states
    for name, masked in forms.items():
        work[name] = dict(zip(("landmarks", "candidates", "inliers"), run(masked, count=True)[3]))
    unmasked = [s for s in range(B) if s not in forms["hood_half"]]
    agree = all(all(np.array_equal(ends["hood_half"][s][k], ends["no_mask"][s][k], equal_nan=True) for k in STATE_KEYS)
                for s in unmasked)
    masked_differ = sum(int(not np.array_equal(ends["hood_all"][s]["keys"], ends["no_mask"][s]["keys"])) for s in range(B))
    line = dict(bench="vo_masks", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup, shape=f"{cols}x{rows}",
                hood_masked_px=int((hood == 0).sum()),
                ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                frames_per_s={k: round(B * 1e3 / min(vs), 1) for k, vs in res.items()},
                bootstrap_ok=boot_ok, final_status_ok={k: sum(int(x["status"] == VOBatch.OK) for x in v) for k, v in ends.items()},
                final_landmarks={k: sum(len(x["lm"]) for x in v) for k, v in ends.items()},
                final_candidates={k: sum(len(x["keys"]) for x in v) for k, v in ends.items()},
                per_step_per_sequence=work, hood_all_sequences_differing=masked_differ,
                hood_half_unmasked_equal_no_mask=bool(agree), **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    assert agree, "an unmasked sequence of hood_half ended differently from no_mask"


if __name__ == "__main__":
    main()
