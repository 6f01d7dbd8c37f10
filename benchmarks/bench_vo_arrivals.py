#!/usr/bin/env python
"""Listed steps of the device-resident loop (VOBatch.step_dev with `seqs`): what a step costs when only some sequences of a
batch have a new frame, and what a fleet of streams at different frame rates costs in one batch.

  python benchmarks/bench_vo_arrivals.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

The workload of bench_vo_frame_size.py: 64 sequences over 16 rendered scenes at KITTI's three native image sizes in
1242 x 376 slots, each with its own frame size and camera, visited forwards and backwards (workload.frame_at), with the
reference's KITTI options.  Every sequence is bootstrapped on the device on frames frame_at(F, k) and frame_at(F, k + 2),
k = s // distinct; its i-th step takes frame_at(F, k + 3 + i).  Frames are resident on the device and submitted one step
ahead.  Forms:

  (a) listed_k    one VOBatch of all sequences; every step lists sequences 0 .. k-1 (k = 1, 8, 32, 64)
  (b) batch_k     a VOBatch of sequences 0 .. k-1 alone, stepped with the plain step
                  (a) - (b) is what the pyramid carry and the unlisted sequences cost
  (c) mixed_rate  one VOBatch of all sequences on a 30 Hz tick: sequences 0-31 every tick, 32-47 every second tick and
                  48-63 every third tick, each tick a listed step of the sequences that have a frame
  (d) per_rate    one VOBatch per rate group, each stepped (plain step) on the ticks of its group

Each run times `--steps` steps (ticks for (c) and (d)) after `--warmup` (wall clock around work that ends in a device
synchronise); the forms alternate.  (c) and (d) must leave every sequence in the same state, array for array; so must (a)
and (b) for the listed sequences.  Prints one JSON line: ms per step (tick), frames per second, whether the states agree,
and the device name, power limit and max SM clock.
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

from bench_vo_frame_size import KITTI, SLOT, group_camera, slot_layout  # noqa: E402
from bench_vo_loop import device_info  # noqa: E402
from mini_vo import REFERENCE_KITTI_OPTIONS as OPT  # noqa: E402

STATE_KEYS = ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses", "status")
KS = (1, 8, 32, 64)


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
    grp = [s % D % 3 for s in range(B)]                       # the KITTI group (size, camera) of sequence s
    scenes = [synth.render_sequence("kitti", F, seed=d, width=KITTI[d % 3][3][1], height=KITTI[d % 3][3][0],
                                    K=group_camera(d % 3))["frames"] for d in range(D)]
    start = [s // D for s in range(B)]
    K_seq = np.stack([group_camera(g) for g in grp])
    sizes = np.int32([KITTI[g][3] for g in grp])
    period = 2 * F - 2
    n_total = args.warmup + args.steps
    img = lambda s, i: scenes[s % D][workload.frame_at(F, start[s] + i)]
    caps = dict(max_landmarks=4096, max_candidates=8192, max_frames=n_total + 8)
    # table[s, j]: sequence s's frame of its j-th step (mod period), slot layout, on the device
    table = torch.from_numpy(np.stack([slot_layout([img(s, 3 + j) for j in range(period)]) for s in range(B)])).cuda()
    rates = [1] * (B // 2) + [2] * (B // 4) + [3] * (B - B // 2 - B // 4)
    rate_groups = [np.flatnonzero(np.int32(rates) == r) for r in (1, 2, 3)]

    def outs(n):
        o = dict(status=torch.zeros(n, dtype=torch.int32, device="cuda"), n_inliers=torch.zeros(n, dtype=torch.int32, device="cuda"),
                 n_lm=torch.zeros(n, dtype=torch.int32, device="cuda"), n_cand=torch.zeros(n, dtype=torch.int32, device="cuda"),
                 pose_cw=torch.zeros((n, 12), dtype=torch.float64, device="cuda"))
        return o, {k: v.data_ptr() for k, v in o.items()}

    def new_batch(members):
        vb = VOBatch(len(members), *SLOT, K_seq[members], OPT, frame_size=sizes[members], **caps)
        r = vb.bootstrap([img(s, 0) for s in members], [img(s, 2) for s in members])
        return vb, int((r["status"] == VOBatch.OK).sum())

    # the ticks of the mixed-rate schedule: the listed sequences and their frames, built on the device before any timing
    ticks, count = [], np.zeros(B, np.int64)
    for t in range(n_total):
        seqs = np.int32([s for s in range(B) if t % rates[s] == 0])
        ticks.append((seqs, table[torch.from_numpy(seqs.astype(np.int64)).cuda(),
                                  torch.from_numpy(count[seqs] % period).cuda()].contiguous()))
        count[seqs] += 1
    listed_sets = {k: [table[:k, j].contiguous() for j in range(period)] for k in KS}
    kept = {}
    torch.cuda.synchronize()

    def timed(steps):
        """steps: callables, one per tick, each enqueueing that tick's submit (one ahead) and step"""
        t0 = None
        for t in range(n_total):
            if t == args.warmup:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            steps(t)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def listed(k):
        vb, ok = new_batch(np.arange(B))
        _, ptr = outs(k)
        seqs = np.arange(k, dtype=np.int32)
        sets = listed_sets[k]
        vb.submit_frames_dev(sets[0].data_ptr(), seqs=seqs)

        def tick(t):
            if t + 1 < n_total:
                vb.submit_frames_dev(sets[(t + 1) % period].data_ptr(), seqs=seqs)
            vb.step_dev(None, ptr, seqs=seqs)
        return timed(tick), [vb.read_state(s) for s in range(k)], ok, [vb]

    def batch_of(k):
        vb, ok = new_batch(np.arange(k))
        _, ptr = outs(k)
        sets = listed_sets[k]
        vb.submit_frames_dev(sets[0].data_ptr())

        def tick(t):
            if t + 1 < n_total:
                vb.submit_frames_dev(sets[(t + 1) % period].data_ptr())
            vb.step_dev(None, ptr)
        return timed(tick), [vb.read_state(s) for s in range(k)], ok, [vb]

    def mixed_rate():
        vb, ok = new_batch(np.arange(B))
        _, ptr = outs(B)
        vb.submit_frames_dev(ticks[0][1].data_ptr(), seqs=ticks[0][0])

        def tick(t):
            if t + 1 < n_total:
                vb.submit_frames_dev(ticks[t + 1][1].data_ptr(), seqs=ticks[t + 1][0])
            vb.step_dev(None, ptr, seqs=ticks[t][0])
        return timed(tick), [vb.read_state(s) for s in range(B)], ok, [vb]

    def per_rate():
        vbs, oks, ptrs, sets = [], 0, [], []
        for r, members in zip((1, 2, 3), rate_groups):
            vb, ok = new_batch(members)
            vbs.append(vb)
            oks += ok
            ptrs.append(outs(len(members))[1])
            m = torch.from_numpy(members.astype(np.int64)).cuda()
            sets.append([table[m, j].contiguous() for j in range(period)])
        torch.cuda.synchronize()
        n_steps = [0, 0, 0]
        for g in range(3):
            vbs[g].submit_frames_dev(sets[g][0].data_ptr())

        def tick(t):
            for g, r in enumerate((1, 2, 3)):
                if t % r:
                    continue
                i = n_steps[g]
                if t + r < n_total:
                    vbs[g].submit_frames_dev(sets[g][(i + 1) % period].data_ptr())
                vbs[g].step_dev(None, ptrs[g])
                n_steps[g] += 1
        el = timed(tick)
        st = [None] * B
        for g, members in enumerate(rate_groups):
            for j, s in enumerate(members):
                st[s] = vbs[g].read_state(j)
        return el, st, oks, vbs

    forms = {f"listed_{k}": (lambda k=k: listed(k)) for k in KS}
    forms.update({f"batch_{k}": (lambda k=k: batch_of(k)) for k in KS})
    forms.update(mixed_rate=mixed_rate, per_rate=per_rate)
    order = [f for k in KS for f in (f"listed_{k}", f"batch_{k}")] + ["mixed_rate", "per_rate"]
    res = {k: [] for k in order}
    boot_ok, ends = {}, {}
    for _ in range(args.runs):
        for name in order:
            el, st, ok, vbs = forms[name]()
            res[name].append(1e3 * el / args.steps)
            boot_ok[name], ends[name] = ok, st
            for vb in vbs:
                vb.close()

    def same(a, b):
        return all(all(np.array_equal(x[k], y[k], equal_nan=True) for k in STATE_KEYS) for x, y in zip(a, b))

    frames_per_tick = sum(len(s) for s, _ in ticks[args.warmup:]) / args.steps
    agree_listed = {k: bool(same(ends[f"listed_{k}"], ends[f"batch_{k}"])) for k in KS}
    agree_rate = bool(same(ends["mixed_rate"], ends["per_rate"]))
    fps = {k: round(k * 1e3 / min(res[f"listed_{k}"]), 1) for k in KS}
    line = dict(bench="vo_arrivals", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup, slot=f"{SLOT[1]}x{SLOT[0]}",
                ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                listed_frames_per_s=fps,
                mixed_rate_frames_per_tick=round(frames_per_tick, 3),
                mixed_rate_frames_per_s={k: round(frames_per_tick * 1e3 / min(res[k]), 1) for k in ("mixed_rate", "per_rate")},
                bootstrap_ok=boot_ok,
                final_status_ok={k: sum(int(x["status"] == VOBatch.OK) for x in v) for k, v in ends.items()},
                listed_equals_batch_of_k=agree_listed, mixed_rate_equals_per_rate=agree_rate, **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")
    assert agree_rate and all(agree_listed.values()), "listed steps and separate batches leave different states"


if __name__ == "__main__":
    main()
