#!/usr/bin/env python
"""The device-resident VO loop (batch.VOBatch) against the loop a user of the batch API writes without it.

  python benchmarks/bench_vo_loop.py [--batch 64] [--distinct 16] [--frames 10] [--steps 150] [--warmup 10] [--runs 2]

64 KITTI-shaped sequences over 16 rendered scenes, visited forwards and backwards (workload.frame_at), with the
reference's KITTI options.  Sequence s uses scene s % distinct and starts at frame s // distinct; it is bootstrapped
once (SIFT + ratio test + findEssentialMat + recoverPose + triangulation, outside the timed region) on that frame and
the one two frames later.  Three forms of the same loop, each from the same bootstrap and over the same frames:

  (a) resident_dev   VOBatch.step_dev, frames resident on the device and submitted one step ahead
  (b) resident_host  VOBatch.step with page-locked host frames
  (c) glued          SequenceBatch.step + numpy compaction + the batched triangulation / detection / distance calls +
                     numpy appends (what tests/mini_vo.py does, batched)

Each run times `--steps` steps after `--warmup` steps (wall clock around work that ends in a device synchronise); the
forms alternate, `--runs` times.  Prints one JSON line: ms per step, frames per second, the per-sequence final
num_pts (inliers of the last step) and n_poses of every form, and the device name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from mini_vo import REFERENCE_KITTI_OPTIONS as OPT, rodrigues  # noqa: E402


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, plim, clk = (v.strip() for v in out.split(","))
        return dict(device=name, power_limit=plim, max_sm_clock=clk)
    except Exception as e:   # the numbers still stand; the card is then named by torch only
        import torch
        return dict(device=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


class Glued:
    """The loop on the batch API without b200vo_loop: numpy state on the host, one synchronous call per stage."""

    def __init__(self, batch, K, states, frames0, L, Cn, P):
        from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch
        o = OPT
        self.K, self.b, self.L, self.Cn, self.P = K, batch, L, Cn, P
        self.sb = SequenceBatch(batch, frames0.shape[1], frames0.shape[2], K, win=o["winSize"], max_level=o["maxLevel"],
                                criteria=o["criteria"], pnp_iters=o["PnP_iterations"], pnp_reproj_err=o["PnP_error"],
                                pnp_conf=o["PnP_conf"], max_landmarks=L, max_candidates=Cn)
        self.sb.prime(frames0)
        self.st = [dict((k, np.asarray(st[k])) for k in ("lm", "lm_kp", "keys", "first_keys", "first_pose", "poses")) for st in states]
        self.live = np.ones(batch, bool)
        self.num_pts = np.zeros(batch, np.int32)
        self.lm_pts = self.sb.pinned_empty((batch, L, 2), np.float32)
        self.lm_obj = self.sb.pinned_empty((batch, L, 3), np.float32)
        self.cand = self.sb.pinned_empty((batch, Cn, 2), np.float32)
        self.n_lm = np.zeros(batch, np.int32)
        self.n_cand = np.zeros(batch, np.int32)

    def step(self, frames):
        from monocular_visual_odometry_va4mr_b200 import hotpath
        o, b, st = OPT, self.b, self.st
        for s in range(b):
            x = st[s]
            n, m = (len(x["lm"]), len(x["keys"])) if self.live[s] else (0, 0)
            self.n_lm[s], self.n_cand[s] = n, m if m > 1 else 0
            if n:
                self.lm_pts[s, :n], self.lm_obj[s, :n] = x["lm_kp"], x["lm"]
            if m > 1:
                self.cand[s, :m] = x["keys"]
        r = self.sb.step(frames, self.lm_pts, self.lm_obj, self.n_lm, self.cand, self.n_cand)
        fk = np.zeros((b, self.Cn, 2), np.float32)
        ky = np.zeros((b, self.Cn, 2), np.float32)
        fp = np.zeros((b, self.Cn), np.int32)
        tri_n = np.zeros(b, np.int32)
        poses = np.zeros((b, self.P, 12))
        n_poses = np.zeros(b, np.int32)
        cur = np.zeros((b, 12))
        for s in range(b):
            if not self.live[s]:
                continue
            x, n = st[s], self.n_lm[s]
            tr = r["lm_status"][s, :n] == 1
            if self.n_cand[s]:
                keep = r["cand_status"][s, :self.n_cand[s]] == 1
                x["keys"], x["first_keys"], x["first_pose"] = r["cand_next"][s, :self.n_cand[s]][keep], x["first_keys"][keep], x["first_pose"][keep]
            if tr.sum() < 8 or not r["pnp_ok"][s]:
                self.live[s] = False
                continue
            inl = r["inlier_mask"][s, :n] == 1
            x["lm"], x["lm_kp"] = x["lm"][inl], r["lm_next"][s, :n][inl]
            self.num_pts[s] = r["n_inliers"][s]
            R_WC = rodrigues(r["pose"][s, :3])
            x["cur"] = np.hstack([R_WC.T.reshape(9), (-R_WC.T @ r["pose"][s, 3:].reshape(3, 1)).reshape(3)])
            m = len(x["keys"])
            if m > 1:
                tri_n[s] = m
                fk[s, :m], ky[s, :m], fp[s, :m] = x["first_keys"], x["keys"], x["first_pose"]
            poses[s, :len(x["poses"])], n_poses[s], cur[s] = x["poses"], len(x["poses"]), x["cur"]
        too_short, new_lm, new_kp, n_new = hotpath.batch_triangulate_landmarks(self.K, o, fk, ky, fp, tri_n, poses, n_poses, cur,
                                                                               ctx=self.sb.ctx)
        corners, n_c = self.sb.good_features(o["feature_max_corners"], o["feature_quality_level"], o["feature_min_dist"])
        existing = np.zeros((b, self.Cn, 2), np.float32)
        m_ex = np.zeros(b, np.int32)
        for s in range(b):
            if not self.live[s]:
                n_c[s] = 0
                continue
            x = st[s]
            if tri_n[s]:
                k = n_new[s]
                if len(x["lm"]) + k > self.L:   # the resident loop stops such a sequence with OVERFLOW
                    self.live[s] = False
                    n_c[s] = 0
                    continue
                x["lm"], x["lm_kp"] = np.concatenate([x["lm"], new_lm[s, :k]]), np.concatenate([x["lm_kp"], new_kp[s, :k]])
                ts = too_short[s, :tri_n[s]]
                x["keys"], x["first_keys"], x["first_pose"] = x["keys"][ts], x["first_keys"][ts], x["first_pose"][ts]
            m_ex[s] = len(x["keys"])
            existing[s, :m_ex[s]] = x["keys"]
        valid = hotpath.batch_min_distance_mask(corners, n_c, existing, m_ex, o["feature_min_dist"], ctx=self.sb.ctx)
        for s in range(b):
            if not self.live[s]:
                continue
            x = st[s]
            c = corners[s, :n_c[s]][valid[s, :n_c[s]]]
            if len(x["keys"]) + len(c) > self.Cn:
                self.live[s] = False
                continue
            x["keys"], x["first_keys"] = np.concatenate([x["keys"], c]), np.concatenate([x["first_keys"], c])
            x["first_pose"] = np.concatenate([x["first_pose"], np.full(len(c), len(x["poses"]), np.int32)])
            x["poses"] = np.vstack([x["poses"], x["cur"]])

    def summary(self):
        return ([int(n) if l else 0 for n, l in zip(self.num_pts, self.live)],
                [len(x["poses"]) if l else 0 for x, l in zip(self.st, self.live)])


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
    from monocular_visual_odometry_va4mr_b200.batch import VOBatch, initial_state, match_bootstrap_frames

    B, D, F = args.batch, args.distinct, args.frames
    scenes = [synth.render_sequence("kitti", F, seed=d)["frames"] for d in range(D)]
    K = synth.SHAPES["kitti"][0].copy()
    rows, cols = scenes[0].shape[1:]
    start = [s // D for s in range(B)]
    states = []
    boot = {}
    for s in range(B):
        d, k = s % D, start[s]
        if (d, k) not in boot:
            f0, f1 = scenes[d][workload.frame_at(F, k)], scenes[d][workload.frame_at(F, k + 2)]
            boot[d, k] = initial_state(K, OPT, *match_bootstrap_frames(f0, f1, OPT["feature_ratio"]))
        states.append(boot[d, k])
    period = 2 * F - 2
    n_total = args.warmup + args.steps
    # the frame set of step t (t = 0, 1, ...): sequence s sees frame frame_at(F, start[s] + 3 + t); sets repeat with `period`
    sets = np.stack([np.stack([scenes[s % D][workload.frame_at(F, start[s] + 3 + t)] for s in range(B)]) for t in range(period)])
    frames0 = np.stack([scenes[s % D][workload.frame_at(F, start[s] + 2)] for s in range(B)])
    L, Cn, P = 4096, 8192, n_total + 8

    def new_loop():
        vb = VOBatch(B, rows, cols, K, OPT, max_landmarks=L, max_candidates=Cn, max_frames=P)
        for s in range(B):
            vb.load(s, frames0[s], states[s])
        return vb

    def final(vb):
        st = [vb.read_state(s) for s in range(B)]
        return [len(x["poses"]) if x["status"] == VOBatch.OK else 0 for x in st], [x["status"] for x in st]

    dev_sets = torch.from_numpy(sets).cuda()
    out = dict(status=torch.zeros(B, dtype=torch.int32, device="cuda"), n_inliers=torch.zeros(B, dtype=torch.int32, device="cuda"),
               n_lm=torch.zeros(B, dtype=torch.int32, device="cuda"), n_cand=torch.zeros(B, dtype=torch.int32, device="cuda"),
               pose_cw=torch.zeros((B, 12), dtype=torch.float64, device="cuda"))
    out_ptr = {k: v.data_ptr() for k, v in out.items()}
    torch.cuda.synchronize()

    def run_dev():
        vb = new_loop()
        vb.submit_frames_dev(dev_sets[0].data_ptr())
        t0 = None
        for t in range(n_total):
            if t == args.warmup:
                vb.ctx.sync()
                t0 = time.perf_counter()
            if t + 1 < n_total:
                vb.submit_frames_dev(dev_sets[(t + 1) % period].data_ptr())
            vb.step_dev(None, out_ptr)
        vb.ctx.sync()
        return time.perf_counter() - t0, vb, out["n_inliers"].cpu().numpy()

    def run_host():
        vb = new_loop()
        pinned = vb.pinned_empty(sets.shape, np.uint8)
        pinned[...] = sets
        t0 = None
        for t in range(n_total):
            if t == args.warmup:
                t0 = time.perf_counter()
            r = vb.step(pinned[t % period])
        dt = time.perf_counter() - t0
        return dt, vb, np.array(r["n_inliers"])

    def run_glued():
        g = Glued(B, K, states, frames0, L, Cn, P)
        t0 = None
        for t in range(n_total):
            if t == args.warmup:
                t0 = time.perf_counter()
            g.step(sets[t % period])
        return time.perf_counter() - t0, g

    res = {k: [] for k in ("resident_dev", "resident_host", "glued")}
    ends = {}
    for _ in range(args.runs):
        for name, fn in (("resident_dev", run_dev), ("resident_host", run_host)):
            dt, vb, n_inl = fn()
            res[name].append(1e3 * dt / args.steps)
            ends[name] = final(vb) + (n_inl.tolist(),)
            vb.close()
        dt, g = run_glued()
        res["glued"].append(1e3 * dt / args.steps)
        ends["glued"] = g.summary()
    num_pts = {k: ends[k][2] for k in ("resident_dev", "resident_host")} | {"glued": ends["glued"][0]}
    n_poses = {k: ends[k][0] for k in ("resident_dev", "resident_host")} | {"glued": ends["glued"][1]}
    agree = all(v == num_pts["glued"] for v in num_pts.values()) and all(v == n_poses["glued"] for v in n_poses.values())
    line = dict(bench="vo_loop", batch=B, distinct=D, frames=F, steps=args.steps, warmup=args.warmup, shape=f"kitti {cols}x{rows}",
                ms_per_step={k: [round(v, 4) for v in vs] for k, vs in res.items()},
                frames_per_s={k: round(B * 1e3 / min(vs), 1) for k, vs in res.items()},
                final_num_pts=num_pts, final_n_poses=n_poses, status_resident=ends["resident_host"][1], forms_agree=bool(agree),
                **device_info())
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "a") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
