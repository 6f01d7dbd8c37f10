#!/usr/bin/env python
"""Benchmark of the per-frame correspondence-and-pose hot path (BASELINE.json metric:
frames/s of KLT + PnP-RANSAC on 1241x376 frames with 2k tracked points).

One *step* = one new frame for each of this rank's synthetic KITTI-shaped sequences: pyramid build,
KLT on ~1000 landmark keypoints and ~1000 candidate keypoints (reference
VisualOdometryPipeLine.py:281,:287), P3P-RANSAC + EPnP on the tracked landmarks (:343).

Headline (BASELINE.json configs[4], SURVEY 8e): `--batch` (64) sequences IN TOTAL, sharded over the
ranks in contiguous blocks with no data-path collective ("scaling": "strong"); the poses are gathered
over NCCL at the end of the timed region.  The fixed-work-per-GPU form (64 sequences on EVERY rank)
is measured too and reported as the named extra `weak_scaling` (`--scaling weak` makes it the headline).

  python bench.py --gpus N --steps K --warmup W            # B200 arm (libb200vo.so)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own cv2 CPU path
  python bench.py --gpus 1 --steps K --dump-outputs DIR    # + the last timed step's results as DIR/<name>.npy

Prints ONE JSON line on rank 0.  Everything that is not the headline (`single_sequence`, `detect`,
`weak_scaling`, `parity`, `cpu_baseline`) is guarded: a failure there is recorded as {"error": ...}
on the line instead of voiding it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "frames/s KLT+PnP-RANSAC 1241x376 2k pts"


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="independent sequences: in total (strong) / per GPU (weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong: --batch sequences sharded over the ranks (BASELINE configs[4]); weak: --batch per rank")
    ap.add_argument("--shape", default="kitti", choices=["kitti", "parking", "malaga"])
    ap.add_argument("--frames", type=int, default=6, help="distinct frames per sequence (visited back and forth)")
    ap.add_argument("--distinct", type=int, default=16, help="distinct rendered scenes the sequences cycle through")
    ap.add_argument("--landmarks", type=int, default=1000)
    ap.add_argument("--candidates", type=int, default=1000)
    ap.add_argument("--cpu-seqs", type=int, default=0, help="sequences per step in the bounded CPU sample (0 = one per host core, at least 4)")
    ap.add_argument("--cpu-steps", type=int, default=10)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-single", action="store_true", help="skip the extra one-sequence-per-call and detection measurements")
    ap.add_argument("--no-weak", action="store_true", help="skip the extra 64-per-GPU (weak scaling) measurement at N > 1")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run oracle check of the last timed step")
    ap.add_argument("--no-lookahead", action="store_true", help="device-resident loop: pass each step's frames with the step instead of one step ahead")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed device-resident step to DIR/<name>.npy (rank 0's sequences)")
    return ap.parse_args(argv)


# ------------------------------------------------------------------------------------------
def clocks_sampler(stop, out, dev):
    """Samples SM clock / throttle reasons DURING the timed regions (NVML; nvidia-smi as a fallback)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
        R = pynvml
        while not stop.is_set():
            sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
            rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
                else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            flags = ["Active" if rs & getattr(R, nm, 0) else "Not Active" for nm in (
                "nvmlClocksThrottleReasonHwSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown",
                "nvmlClocksThrottleReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwPowerCap")]
            out.append([str(sm), str(mx), "0", hex(rs)] + flags)
            stop.wait(0.02)
        return
    except Exception:
        pass
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", f"--id={dev}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            if r.returncode == 0 and r.stdout.strip():
                out.append([c.strip() for c in r.stdout.strip().splitlines()[0].split(",")])
        except Exception:
            pass
        stop.wait(0.2)


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = [float(s[0]) for s in samples if s[0].replace(".", "").isdigit()]
    mx = [float(s[1]) for s in samples if s[1].replace(".", "").isdigit()]
    reasons = set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for s in samples:
        for k, nm in enumerate(names):
            if len(s) > 4 + k and s[4 + k].lower().startswith("active"):
                reasons.add(nm)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(samples)}


def pin_to_gpu_cores(dev):
    """Restrict this rank to the CPU cores NVML lists as local to its GPU (first-touch then places the rank's
    page-locked buffers on that NUMA node).  -> number of cores, or None when NVML has no answer."""
    import pynvml
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(dev)
    n_words = (os.cpu_count() + 63) // 64
    mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
    cores = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
    cores = [c for c in cores if c in os.sched_getaffinity(0)]
    if not cores:
        return None
    os.sched_setaffinity(0, cores)
    return len(cores)


def guarded(fn, *a, **kw):
    """Run a non-headline measurement; a failure becomes {"error": ...} on the JSON line."""
    try:
        return fn(*a, **kw)
    except BaseException as e:  # noqa: BLE001 -- the headline must print whatever an extra does
        if isinstance(e, KeyboardInterrupt):
            raise
        tb = traceback.format_exc().strip().splitlines()
        return {"error": f"{type(e).__name__}: {e}", "where": tb[-3:] if len(tb) >= 3 else tb}


def spread(ms):
    """min / median / max of a list of per-step times (ms)."""
    if not len(ms):
        return None
    a = np.asarray(ms, np.float64)
    return {"min": float(a.min()), "median": float(np.median(a)), "max": float(a.max()), "n": int(a.size)}


def cpu_reference_step(cv2, wl, opts, f, g, seqs):
    """The reference's own cv2 calls for one frame of each sequence in `seqs` (VisualOdometryPipeLine.py
    :281, :287, :343 with its KITTI options)."""
    n = 0
    for s in seqs:
        nl, nc = int(wl.n_lm[f, s]), int(wl.n_cand[f, s])
        prev, nxt = wl.frames[f, s], wl.frames[g, s]
        p, st, _ = cv2.calcOpticalFlowPyrLK(prev, nxt, wl.lm_pts[f, s, :nl], None, winSize=opts["win"],
                                            maxLevel=opts["max_level"], criteria=opts["criteria"])
        keep = (st == 1).squeeze()
        if nc > 1:
            cv2.calcOpticalFlowPyrLK(prev, nxt, wl.cand_pts[f, s, :nc], None, winSize=opts["win"],
                                     maxLevel=opts["max_level"], criteria=opts["criteria"])
        kp, lm = p[keep], wl.lm_obj[f, s, :nl][keep]
        if len(kp) >= 8:
            cv2.solvePnPRansac(lm, kp, wl.K, np.zeros(4), flags=cv2.SOLVEPNP_P3P, confidence=opts["pnp_conf"],
                               reprojectionError=opts["pnp_err"], iterationsCount=opts["pnp_iters"])
        n += 1
    return n


def time_cpu_reference(wl, opts, n_seqs, steps, warmup):
    """-> (frames/s, cores, kind, sample description).  cv2 is the reference's own CPU implementation of the
    path; two ways of using all host threads are timed and the FASTER one is reported: (a) the reference as
    written -- sequences one after the other, cv2's internal parallel_for over all cores; (b) one thread per
    sequence (cv2 releases the GIL), cv2 single-threaded inside.  If cv2 is not importable the C oracle port is
    timed instead (kind 'port', 1 core)."""
    from concurrent.futures import ThreadPoolExecutor
    from monocular_visual_odometry_va4mr_b200 import workload
    fo = lambda t: workload.frame_at(wl.F, t)
    seqs = list(range(min(n_seqs, wl.batch)))
    steps = max(int(steps), 1)
    try:
        import cv2
    except ImportError:
        cv2 = None
    if cv2 is not None:
        cores = os.cpu_count() or 1

        def run(mode):
            if mode == "internal":
                cv2.setNumThreads(cores)
                step = lambda f, g: cpu_reference_step(cv2, wl, opts, f, g, seqs)
            else:
                cv2.setNumThreads(1)
                pool = ThreadPoolExecutor(max_workers=cores)
                step = lambda f, g: sum(pool.map(lambda s_: cpu_reference_step(cv2, wl, opts, f, g, [s_]), seqs))
            for t in range(warmup):
                step(fo(t), fo(t + 1))
            t0 = time.perf_counter()
            n = 0
            for t in range(warmup, warmup + steps):
                n += step(fo(t), fo(t + 1))
            return n / (time.perf_counter() - t0)

        fps_a, fps_b = run("internal"), run("pool")
        cv2.setNumThreads(cores)
        mode = "cv2 internal threading" if fps_a >= fps_b else "one thread per sequence"
        return max(fps_a, fps_b), cores, "reference", (
            f"cv2 {cv2.__version__} calcOpticalFlowPyrLK x2 + solvePnPRansac(P3P), {len(seqs)} sequences x {steps} frames, "
            f"{cores} threads; best of cv2-internal threading ({fps_a:.0f} f/s) and one thread per sequence ({fps_b:.0f} f/s): {mode}")
    import oracle
    t0 = time.perf_counter()
    n = 0
    for t in range(steps):
        f, g = fo(t), fo(t + 1)
        for s in seqs:
            nl, nc = int(wl.n_lm[f, s]), int(wl.n_cand[f, s])
            p, st, _ = oracle.calc_optical_flow_pyr_lk(wl.frames[f, s], wl.frames[g, s], wl.lm_pts[f, s, :nl],
                                                       opts["win"], opts["max_level"], opts["criteria"])
            oracle.calc_optical_flow_pyr_lk(wl.frames[f, s], wl.frames[g, s], wl.cand_pts[f, s, :nc],
                                            opts["win"], opts["max_level"], opts["criteria"])
            keep = st.ravel() == 1
            oracle.solve_pnp_ransac_p3p(wl.lm_obj[f, s, :nl][keep], p[keep], wl.K, opts["pnp_iters"], opts["pnp_err"], opts["pnp_conf"])
            n += 1
    dt = time.perf_counter() - t0
    return n / dt, 1, "port", f"C oracle port, {len(seqs)} sequences x {steps} frames, 1 thread"


def caps(args):
    return (1024 if args.landmarks <= 1024 else args.landmarks), (1024 if args.candidates <= 1024 else args.candidates)


def make_workload(args, n_seq, first_index):
    from monocular_visual_odometry_va4mr_b200 import workload
    capL, capC = caps(args)
    return workload.TrackWorkload(args.shape, batch=n_seq, n_frames=args.frames, n_landmarks=args.landmarks,
                                  n_candidates=args.candidates, n_distinct=max(1, args.distinct), seed=0,
                                  cap_landmarks=capL, cap_candidates=capC, first_index=first_index)


def shard_plan(total, world, rank, scaling):
    """-> (first global sequence index, sequences on this rank, sequences in the whole job)."""
    from monocular_visual_odometry_va4mr_b200 import sharding
    if scaling == "weak":
        return rank * total, total, world * total
    lo, hi = sharding.shard_range(total, world, rank)
    return lo, hi - lo, total


def pyramid_pixels(wl, opts):
    levels, w_, h_ = 1, wl.w, wl.h
    P = w_ * h_
    for _ in range(opts["max_level"]):
        w_, h_ = (w_ + 1) // 2, (h_ + 1) // 2
        if w_ <= opts["win"][0] or h_ <= opts["win"][1]:
            break
        P += w_ * h_
        levels += 1
    return P, levels


# ------------------------------------------------------------------------------------------
class Arm:
    """One sharded measurement on this rank: the device-resident loop and the two host-buffer loops."""

    def __init__(self, args, opts, ctx, wl, world, local, total_seqs):
        import torch
        from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch
        self.args, self.opts, self.ctx, self.wl, self.world, self.local, self.total = args, opts, ctx, wl, world, local, total_seqs
        self.torch = torch
        self.dev = torch.device("cuda", local)
        self.sb = SequenceBatch(wl.batch, wl.h, wl.w, wl.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                                pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                                max_landmarks=wl.L, max_candidates=wl.Cn, ctx=ctx)
        self.stream = torch.cuda.ExternalStream(ctx.stream(), device=self.dev)
        self.K, self.W = max(args.steps, 1), max(args.warmup, 3)

    def fo(self, t):
        from monocular_visual_odometry_va4mr_b200 import workload
        return workload.frame_at(self.wl.F, t)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize()
        self.ctx.sync()

    def max_over_ranks(self, vals):
        if self.world == 1:
            return [float(v) for v in vals]
        import torch.distributed as dist
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    # ---- (1) device-resident: every input already in HBM ----
    def device_resident(self, gather_counts):
        torch, wl, sb, ctx, K, W = self.torch, self.wl, self.sb, self.ctx, self.K, self.W
        from monocular_visual_odometry_va4mr_b200 import _lib, sharding
        dev = self.dev
        P = min(K, 50)     # steps of the separate, profiled pass behind the timed region (stage times for the roofline)
        d_frames = torch.from_numpy(wl.frames).to(dev)
        d_lm_pts = torch.from_numpy(wl.lm_pts).to(dev)
        d_lm_obj = torch.from_numpy(wl.lm_obj).to(dev)
        d_n_lm = torch.from_numpy(wl.n_lm).to(dev)
        d_cand = torch.from_numpy(wl.cand_pts).to(dev)
        d_n_cand = torch.from_numpy(wl.n_cand).to(dev)
        b, L, Cn = wl.batch, wl.L, wl.Cn
        d_out = dict(lm_next=torch.zeros((b, L, 2), dtype=torch.float32, device=dev), lm_status=torch.zeros((b, L), dtype=torch.uint8, device=dev),
                     cand_next=torch.zeros((b, Cn, 2), dtype=torch.float32, device=dev), cand_status=torch.zeros((b, Cn), dtype=torch.uint8, device=dev),
                     pose=torch.zeros((K + W + P, b, 6), dtype=torch.float64, device=dev), pnp_ok=torch.zeros((b,), dtype=torch.uint8, device=dev),
                     inlier_mask=torch.zeros((b, L), dtype=torch.uint8, device=dev), n_inliers=torch.zeros((b,), dtype=torch.int32, device=dev))
        torch.cuda.synchronize()

        ahead = not self.args.no_lookahead

        # raw device addresses, taken once: at 8 sequences per GPU a step is 0.23 ms, and a dozen tensor views +
        # .data_ptr() calls per step (8 ranks sharing one host) made the Python loop, not the GPU, the limit
        F = d_frames.shape[0]
        p_frames = [d_frames[i].data_ptr() for i in range(F)]
        p_in = [(d_lm_pts[i].data_ptr(), d_lm_obj[i].data_ptr(), d_n_lm[i].data_ptr(), d_cand[i].data_ptr(), d_n_cand[i].data_ptr())
                for i in range(F)]
        p_out = {k: v.data_ptr() for k, v in d_out.items()}
        p_pose = [d_out["pose"][t].data_ptr() for t in range(K + W + P)]

        def dev_step(t):
            # look-ahead form (default): the frames of step t+1 were handed over one step earlier
            # (b200vo_batch_submit_frames_dev), so their pyramids are built beside step t-1's pose chain -- what the
            # streaming host API does with b200vo_batch_submit_frames; every input is resident in HBM either way
            f = self.fo(t)
            p_out["pose"] = p_pose[t]
            if ahead:
                sb.submit_frames_dev(p_frames[self.fo(t + 2)])
            sb.step_dev(None if ahead else p_frames[self.fo(t + 1)], *p_in[f], p_out)

        def gather():
            # poses of every rank's sequences over NCCL (padded when the shards are ragged)
            self.stream.synchronize()
            traj = d_out["pose"][:K + W].permute(1, 0, 2).contiguous()       # [sequence, step, 6]
            g = sharding.gather_trajectories(traj, self.world, gather_counts)
            torch.cuda.current_stream().synchronize()
            return g

        sb.prime(wl.frames[self.fo(0)])
        if ahead:
            sb.submit_frames_dev(d_frames[self.fo(1)].data_ptr())
        for t in range(W):
            dev_step(t)
        if self.world > 1:   # the gather of the timed region runs once untimed first (NCCL sets its channels up lazily)
            gather()
        self.barrier()
        launches0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        for t in range(W, W + K):
            dev_step(t)
        gathered = gather() if self.world > 1 else None
        e1.record(self.stream)
        self.barrier()
        dev_ms = e0.elapsed_time(e1)
        launches = ctx.launch_count() - launches0
        # the results of the last timed step, read before the profiled pass below overwrites the output buffers
        timed_last = ({k: (v[W + K - 1] if k == "pose" else v).cpu().numpy() for k, v in d_out.items()}
                      if self.args.dump_outputs else None)
        # Per-launch stage times come from a SEPARATE pass of P more steps right behind the timed region: the timing events
        # b200vo_batch_profile puts between the launches stall this stream structure by ~0.1 ms in every other step (measured
        # with the kernels' own %globaltimer stamps, B200VO_TRACE_FILE: gaps of 8-10 us between launches without them, 100-145
        # with them), so the timed region runs without them.
        ctx.lib.b200vo_batch_profile(sb.h, 1)
        for t in range(W + K, W + K + P):
            dev_step(t)
        self.stream.synchronize()
        stage_ms = np.zeros(3, np.float32)
        nprof = np.zeros(1, np.int32)
        ctx.lib.b200vo_batch_profile_read(sb.h, stage_ms.ctypes.data_as(_lib.c_f32p), nprof.ctypes.data_as(_lib.c_intp))
        ctx.lib.b200vo_batch_profile(sb.h, 0)
        n_ok = int(d_out["pnp_ok"].sum().item())
        dev_ms = self.max_over_ranks([dev_ms])[0]
        n_gathered = None if gathered is None else int(sum(int(g_.shape[0]) for g_ in gathered))
        last = {k: (v[W + K + P - 1] if k == "pose" else v).cpu().numpy() for k, v in d_out.items()}
        return {"dev_ms": dev_ms, "launches": int(launches), "stage_ms": stage_ms, "nprof": int(nprof[0]), "n_ok": n_ok,
                "gathered_sequences": n_gathered, "last": last, "last_t": W + K + P - 1, "profiled_steps": P,
                "timed_last": timed_last, "timed_last_t": W + K - 1}

    # ---- (2) end to end through the C-ABI with HOST buffers (pinned; H2D + D2H inside the timed region) ----
    def host_buffers(self):
        wl, sb = self.wl, self.sb
        if not hasattr(self, "_h"):
            h_frames = sb.pinned_frames(wl.F)
            h_frames[:] = wl.frames
            self._h = (h_frames, sb.pinned_like(wl.lm_pts), sb.pinned_like(wl.lm_obj), sb.pinned_like(wl.n_lm),
                       sb.pinned_like(wl.cand_pts), sb.pinned_like(wl.n_cand))
        return self._h

    def timed_host_loop(self, prefetch):
        """K steps through b200vo_batch_step with host buffers.  prefetch: the frames of step t+1 are handed to
        b200vo_batch_submit_frames before step t is called (what a video reader does), so their upload and
        pyramid build overlap step t's kernels; every step still uploads one frame set and its point arrays and
        reads every result back inside the timed region.  -> (seconds, per-step wall ms, per-step device ms)."""
        sb, ctx, K, W, fo = self.sb, self.ctx, self.K, self.W, self.fo
        h_frames, h_lm_pts, h_lm_obj, h_n_lm, h_cand, h_n_cand = self.host_buffers()
        sb.prime(h_frames[fo(0)])
        if prefetch:
            sb.submit_frames(h_frames[fo(1)])
        wall, devms = [], []
        t0 = time.perf_counter()
        for t in range(W + K):
            if t == W:
                self.barrier()
                t0 = time.perf_counter()
            ts = time.perf_counter()
            f, g = fo(t), fo(t + 1)
            if prefetch:
                sb.submit_frames(h_frames[fo(t + 2)])
                sb.step(None, h_lm_pts[f], h_lm_obj[f], h_n_lm[f], h_cand[f], h_n_cand[f])
            else:
                sb.step(h_frames[g], h_lm_pts[f], h_lm_obj[f], h_n_lm[f], h_cand[f], h_n_cand[f])
            if t >= W:
                wall.append(1e3 * (time.perf_counter() - ts))
                devms.append(ctx.last_gpu_ms())
        self.barrier()
        dt = time.perf_counter() - t0
        if prefetch:     # consume the frame set submitted ahead of the last timed step
            f = fo(W + K)
            sb.step(None, h_lm_pts[f], h_lm_obj[f], h_n_lm[f], h_cand[f], h_n_cand[f])
        return dt, wall, devms

    def h2d_bandwidth(self, nbytes=64 << 20):
        """Page-locked host -> device copy bandwidth of this rank's link (GB/s, best of 5, CUDA events): the ceiling of
        the end-to-end form, whose every step uploads one frame set."""
        torch = self.torch
        h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        d = torch.empty(nbytes, dtype=torch.uint8, device=self.dev)
        best = 0.0
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            d.copy_(h, non_blocking=True)
            e1.record()
            e1.synchronize()
            best = max(best, nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9)
        return best

    def e2e(self):
        K = self.K
        sync_s, sync_wall, _ = self.timed_host_loop(False)
        s, wall, devms = self.timed_host_loop(True)
        s_local = s
        s, sync_s = self.max_over_ranks([s, sync_s])
        h2d, d2h = self.wl.bytes_per_step()
        link = guarded(self.h2d_bandwidth)
        pcie = None
        if isinstance(link, float) and link > 0:
            pcie = {"h2d_gbs_measured": link, "h2d_gbs_achieved": h2d / (s_local / K) / 1e9, "frac": h2d / (s_local / K) / 1e9 / link,
                    "note": "rank 0's link: bytes uploaded per step / end-to-end step time, against a plain 64 MiB page-locked copy; "
                            "near 1 means the end-to-end form is bound by the host link, not by the kernels"}
        return {"value": self.total * K / s, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "host_link": pcie,
                "ms_per_step": 1e3 * s / K, "host_ms_per_step": spread(wall), "device_ms_per_step": spread(devms),
                "api": "b200vo_batch_submit_frames(t+1) + b200vo_batch_step(t): page-locked host buffers in and out, "
                       "next frames uploaded while the current step runs; per-step spread = wall clock around each call on rank 0, "
                       "device = CUDA events around the call's stream work",
                "call_by_call": {"value": self.total * K / sync_s, "ms_per_step": 1e3 * sync_s / K, "host_ms_per_step": spread(sync_wall),
                                 "api": "b200vo_batch_step(frames) only: upload, kernels and read-back serialised per call"}}

    def close(self):
        self.sb.close()


def parity_check(arm, res, n_check=2):
    """AFTER the timed region: sequences of the LAST timed device-resident step against the CPU oracle
    (oracle/ = test infrastructure; this is the checker, never the thing measured).  KLT: status identical and
    positions bit-equal; PnP: inlier mask identical, pose within 1e-6."""
    import oracle
    wl, opts, last = arm.wl, arm.opts, res["last"]
    t = res["last_t"]
    f, g = arm.fo(t), arm.fo(t + 1)
    seqs = sorted({0, wl.batch - 1} if n_check >= 2 else {0})
    out = {"sequences_checked": len(seqs), "step": int(t), "against": "oracle/ (C restatement pinned to cv2)"}
    ok_all = True
    max_d, pose_d = 0.0, 0.0
    for s in seqs:
        nl, nc = int(wl.n_lm[f, s]), int(wl.n_cand[f, s])
        rp, rst, _ = oracle.calc_optical_flow_pyr_lk(wl.frames[f, s], wl.frames[g, s], wl.lm_pts[f, s, :nl], opts["win"],
                                                     opts["max_level"], opts["criteria"])
        st = last["lm_status"][s, :nl]
        same_st = np.array_equal(st, rst.ravel())
        keep = rst.ravel() == 1
        d = float(np.abs(last["lm_next"][s, :nl][keep] - rp[keep]).max()) if keep.any() else 0.0
        max_d = max(max_d, d)
        ok_s = same_st and d == 0.0
        if nc > 0:
            cp, cst, _ = oracle.calc_optical_flow_pyr_lk(wl.frames[f, s], wl.frames[g, s], wl.cand_pts[f, s, :nc], opts["win"],
                                                         opts["max_level"], opts["criteria"])
            ck = cst.ravel() == 1
            ok_s = ok_s and np.array_equal(last["cand_status"][s, :nc], cst.ravel())
            if ck.any():
                dc = float(np.abs(last["cand_next"][s, :nc][ck] - cp[ck]).max())
                max_d = max(max_d, dc)
                ok_s = ok_s and dc == 0.0
        obj, img = wl.lm_obj[f, s, :nl][keep], np.ascontiguousarray(rp[keep], np.float32)
        if len(obj) >= 4:
            rok, rrv, rtv, rinl, _ = oracle.solve_pnp_ransac_p3p(obj, img, wl.K, opts["pnp_iters"], opts["pnp_err"], opts["pnp_conf"])
            ok_s = ok_s and bool(last["pnp_ok"][s]) == bool(rok)
            if rok:
                want = np.zeros(wl.L, np.uint8)
                want[np.flatnonzero(keep)[np.asarray(rinl).ravel()]] = 1
                ok_s = ok_s and np.array_equal(last["inlier_mask"][s], want) and int(last["n_inliers"][s]) == int(want.sum())
                pd = float(np.abs(last["pose"][s] - np.concatenate([np.ravel(rrv), np.ravel(rtv)])).max())
                pose_d = max(pose_d, pd)
                ok_s = ok_s and pd <= 1e-6 * max(1.0, float(np.abs(rtv).max()))
        ok_all = ok_all and bool(ok_s)
    out.update(ok=bool(ok_all), klt_max_abs_diff_px=max_d, pose_max_abs_diff=pose_d)
    return out


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(arm, res, out_dir):
    """Writes what the last timed device-resident step returned to out_dir/<name>.npy (float32, pose float64), so that
    two builds run with the same arguments can be compared output for output.  Point slots at or past a sequence's
    point count hold no result and are written as 0; sequence_index is each row's global sequence index.  Above
    DUMP_BYTES in all, a fixed seeded sample of the sequences is written."""
    wl, last = arm.wl, res["timed_last"]
    f = arm.fo(res["timed_last_t"])
    lm_live = np.arange(wl.L)[None, :] < wl.n_lm[f][:, None]
    cand_live = np.arange(wl.Cn)[None, :] < wl.n_cand[f][:, None]
    out = {"lm_next": np.where(lm_live[..., None], last["lm_next"], 0).astype(np.float32),
           "lm_status": np.where(lm_live, last["lm_status"], 0).astype(np.float32),
           "cand_next": np.where(cand_live[..., None], last["cand_next"], 0).astype(np.float32),
           "cand_status": np.where(cand_live, last["cand_status"], 0).astype(np.float32),
           "pose": last["pose"].astype(np.float64),
           "pnp_ok": last["pnp_ok"].astype(np.float32),
           "inlier_mask": np.where(lm_live, last["inlier_mask"], 0).astype(np.float32),
           "n_inliers": last["n_inliers"].astype(np.float32),
           "sequence_index": np.arange(wl.first_index, wl.first_index + wl.batch, dtype=np.float64)}
    per_sequence = sum(a.nbytes for a in out.values()) / wl.batch
    keep = int((DUMP_BYTES - 128 * len(out)) // per_sequence)      # 128: header of one .npy file
    if keep < wl.batch:
        rows = np.sort(np.random.default_rng(0).choice(wl.batch, keep, replace=False))
        out = {k: a[rows] for k, a in out.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def measure_detect(arm):
    """extra: Shi-Tomasi detection (reference :256; feature_adding runs it every frame) for the whole batch on
    the resident frames."""
    sb, wl, args = arm.sb, arm.wl, arm.args
    sb.good_features(1400, 0.1, 10.0)
    t0 = time.perf_counter()
    for _ in range(20):
        sb.good_features(1400, 0.1, 10.0)
    dt = (time.perf_counter() - t0) / 20
    detect = {"ms_per_step": 1e3 * dt, "frames_per_s": wl.batch / dt,
              "what": f"b200vo_batch_good_features(1400, 0.1, 10) on the {wl.batch} resident frames, corner lists read back to the host"}
    if not args.no_cpu_baseline:
        try:
            import cv2
        except ImportError:
            return detect
        from concurrent.futures import ThreadPoolExecutor
        cores = os.cpu_count() or 1
        cv2.setNumThreads(1)
        imgs = [wl.frames[0, s_ % wl.batch] for s_ in range(cores)]
        with ThreadPoolExecutor(max_workers=cores) as pool:
            list(pool.map(lambda im: cv2.goodFeaturesToTrack(im, 1400, 0.1, 10, blockSize=3), imgs))
            t0 = time.perf_counter()
            for _ in range(5):
                list(pool.map(lambda im: cv2.goodFeaturesToTrack(im, 1400, 0.1, 10, blockSize=3), imgs))
            detect["cv2_frames_per_s"] = 5 * len(imgs) / (time.perf_counter() - t0)
        cv2.setNumThreads(cores)
        detect["cv2_what"] = f"cv2.goodFeaturesToTrack, one thread per image on {cores} cores"
    return detect


def measure_bootstrap(args):
    """extra: the bootstrap of `initialization` (reference :293-323) from two raw frames -- SIFT detectAndCompute x2
    (:226-227), knnMatch(k=2) + ratio test (:229, :218-224), findEssentialMat (:308), recoverPose (:315) -- on the CUDA
    path through the cv2-shaped shim, and the same calls on cv2.  BASELINE config 2's call chain at the frame's own
    keypoint count (the 8192 x 8192 matcher stress is benchmarks/bench_components.py)."""
    import numpy as np
    from monocular_visual_odometry_va4mr_b200 import cv2_compat, synth, workload
    shape = args.shape
    s = synth.render_sequence(shape, 3, seed=2)
    f0, f1, K = s["frames"][0], s["frames"][2], s["K"]          # main.py:18 bootstrap_frames = [0, 2]

    def chain(m):
        sift = m.SIFT_create()
        k0, d0 = sift.detectAndCompute(f0, None)
        k1, d1 = sift.detectAndCompute(f1, None)
        matches = m.BFMatcher().knnMatch(d0, d1, k=2)
        good = [a for a, b in matches if a.distance < 0.8 * b.distance]
        p0 = np.float32([k0[a.queryIdx].pt for a in good]).reshape(-1, 2)
        p1 = np.float32([k1[a.trainIdx].pt for a in good]).reshape(-1, 2)
        E, mask = m.findEssentialMat(p0, p1, K, method=m.RANSAC, prob=0.99, threshold=1.0)
        n, R, t, _ = m.recoverPose(E, p0[mask.ravel() == 1], p1[mask.ravel() == 1], K)
        return len(k0), len(k1), len(good), int(mask.sum()), int(n)

    def timed(m, reps):
        chain(m)
        t0 = time.perf_counter()
        for _ in range(reps):
            out = chain(m)
        return 1e3 * (time.perf_counter() - t0) / reps, out

    ms, out = timed(cv2_compat, 5)
    boot = {"ms": ms, "keypoints": list(out[:2]), "ratio_test_survivors": out[2], "essential_inliers": out[3], "recover_pose_good": out[4],
            "what": f"{shape}-shaped bootstrap from two raw frames: SIFT x2, knnMatch + ratio test, findEssentialMat, recoverPose through cv2_compat "
                    "(host buffers in and out per call, Python objects for keypoints and matches included)"}
    if not args.no_cpu_baseline:
        try:
            import cv2
        except ImportError:
            return boot
        cv2.setNumThreads(os.cpu_count() or 1)
        cms, cout = timed(cv2, 2)
        boot.update(cv2_ms=cms, x_cv2=cms / ms, cv2_counts=list(cout),
                    cv2_what=f"cv2 {cv2.__version__}, same calls, cv2-internal threading on {os.cpu_count()} cores")
    return boot


def single_plan(K, W):
    """Step counts of the one-sequence extra: (GPU timed steps, cv2 warm-up steps, cv2 timed steps).  Frames are
    addressed with workload.frame_at(), which is defined for every t, so no count can index out of range."""
    return max(1, min(int(K), 200)), 3, 30


def measure_single(args, opts, ctx, W):
    """extra: ONE sequence per call -- BASELINE config 0's shape, latency-bound (frame i needs frame i-1)."""
    from monocular_visual_odometry_va4mr_b200 import workload
    from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch
    n1, cw, nc1 = single_plan(args.steps, W)
    wl1 = make_workload(args, 1, 0)
    fo = lambda t: workload.frame_at(wl1.F, t)
    sb1 = SequenceBatch(1, wl1.h, wl1.w, wl1.K, win=opts["win"], max_level=opts["max_level"], criteria=opts["criteria"],
                        pnp_iters=opts["pnp_iters"], pnp_reproj_err=opts["pnp_err"], pnp_conf=opts["pnp_conf"],
                        max_landmarks=wl1.L, max_candidates=wl1.Cn, ctx=ctx)
    try:
        f1 = sb1.pinned_frames(wl1.F)
        f1[:] = wl1.frames
        a1 = [sb1.pinned_like(x) for x in (wl1.lm_pts, wl1.lm_obj, wl1.n_lm, wl1.cand_pts, wl1.n_cand)]
        sb1.prime(f1[fo(0)])
        sb1.submit_frames(f1[fo(1)])
        wall = []
        t0 = time.perf_counter()
        for t in range(W + n1):
            if t == W:
                ctx.sync()
                t0 = time.perf_counter()
            ts = time.perf_counter()
            sb1.submit_frames(f1[fo(t + 2)])
            f = fo(t)
            sb1.step(None, a1[0][f], a1[1][f], a1[2][f], a1[3][f], a1[4][f])
            if t >= W:
                wall.append(1e3 * (time.perf_counter() - ts))
        dt1 = time.perf_counter() - t0
        f = fo(W + n1)
        sb1.step(None, a1[0][f], a1[1][f], a1[2][f], a1[3][f], a1[4][f])
        single = {"value": n1 / dt1, "unit": "frames/s", "ms_per_frame": 1e3 * dt1 / n1, "frames": n1, "ms_per_frame_spread": spread(wall),
                  "what": "one sequence per b200vo_batch_step call (batch = 1), host buffers in and out, next frame prefetched: "
                          "the latency-bound shape of BASELINE config 0; a single sequence cannot be sharded (frame i needs frame i-1)"}
    finally:
        sb1.close()
    if not args.no_cpu_baseline:
        try:
            import cv2
        except ImportError:
            return single
        cv2.setNumThreads(os.cpu_count() or 1)
        for t in range(cw):
            cpu_reference_step(cv2, wl1, opts, fo(t), fo(t + 1), [0])
        t0 = time.perf_counter()
        for t in range(cw, cw + nc1):
            cpu_reference_step(cv2, wl1, opts, fo(t), fo(t + 1), [0])
        single["cv2_value"] = nc1 / (time.perf_counter() - t0)
        single["x_cv2"] = single["value"] / single["cv2_value"]
        single["cv2_what"] = f"cv2 {cv2.__version__}, same calls, one sequence, cv2-internal threading on {os.cpu_count()} cores"
    return single


def klt_roofline(args, opts, wl, res, roofline_note):
    """Roofline of the dominant kernel (the LANDMARK launch of klt_kernel_v3), timed live with CUDA events on the
    stream it is launched on (b200vo_batch_profile) in a pass of the same loop behind the timed region."""
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    P, levels = pyramid_pixels(wl, opts)
    n_pts_total = int(wl.n_lm[0].sum())
    klt_bytes = wl.batch * 2 * P + n_pts_total * 21           # both pyramids once + this launch's points in/out
    nprof = max(res["nprof"], 1)
    klt_ms = float(res["stage_ms"][1]) / nprof
    achieved = klt_bytes / (klt_ms * 1e-3) / 1e9 if klt_ms > 0 else 0.0
    # measured DRAM traffic of that kernel (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum per launch):
    # taken from the committed capture when it was made on this very workload, else null
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "klt_dram_traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get("workload") == {"shape": args.shape, "batch": wl.batch, "landmarks": args.landmarks, "candidates": args.candidates}:
            traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], tj["source"]
    return {"bound": "hbm", "kernel": "klt_kernel_v3 (landmark launch)", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": klt_bytes, "avg_launch_ms": klt_ms,
            "avg_launch_ms_source": f"CUDA events on the launching stream over {res.get('profiled_steps', 0)} steps of the same loop run right behind "
                                    "the timed region (timing events between the launches stall the timed loop itself by 2-12 %)",
            "stage_ms_per_step": {"pyramid": float(res["stage_ms"][0]) / nprof, "klt_landmarks": klt_ms,
                                  "pose_chain_beside_klt_candidates": float(res["stage_ms"][2]) / nprof,
                                  "pose_stage_note": "event behind the pose kernel, stamped when its stream is serviced again; on the kernels' own "
                                                     "clock (B200VO_TRACE_FILE) the pose CTAs finish 0.14 ms after the landmark launch at 64 sequences"},
            "note": roofline_note}, levels


ROOFLINE_NOTE = ("klt_kernel_v3 is instruction-issue bound (integer bilinear taps from shared-memory-staged windows, ~25 window passes per "
                 "point); its DRAM traffic ~ the algorithmic bytes, so the HBM fraction stays at percent level by construction; see DESIGN.md section 4")


# ------------------------------------------------------------------------------------------
def main(argv=None):
    args = parse(argv)
    if args.cpu_seqs <= 0:
        args.cpu_seqs = max(4, os.cpu_count() or 1)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    from monocular_visual_odometry_va4mr_b200 import workload
    opts = workload.REFERENCE_OPTIONS[args.shape]
    first, n_local, total = shard_plan(args.batch, world, rank, args.scaling)
    how = (f"{args.batch} independent synthetic {args.shape}-shaped sequences in total, sharded over the GPUs in contiguous blocks"
           if args.scaling == "strong" else f"{args.batch} independent synthetic {args.shape}-shaped sequences per GPU")
    cfg_common = {
        "workload": f"{how} (BASELINE.json configs[4] = 64 x the configs[0] sequence shape; SURVEY's C5 = 64 x C1), "
                    f"one new frame each per step: KLT {opts['win'][0]}x{opts['win'][1]} maxLevel {opts['max_level']} criteria {opts['criteria']} on "
                    f"~{args.landmarks} landmark + ~{args.candidates} candidate keypoints, P3P-RANSAC {opts['pnp_iters']} it / {opts['pnp_err']} px + EPnP",
        "shape": args.shape, "sequences_total": total, "landmarks": args.landmarks, "candidates": args.candidates,
        "l2": f"inputs larger than L2 at 64 sequences per GPU ({args.frames} frame sets x sequences rotate through HBM); smaller shards fit L2 and say so in sequences_per_gpu",
    }

    # ---------------- reference arm: the reference's cv2 CPU path, rank 0 only ----------------
    if args.impl == "reference":
        if rank != 0:
            return
        saved = args.distinct
        args.distinct = min(args.distinct, max(2, args.cpu_seqs))
        wl = make_workload(args, args.cpu_seqs, 0)
        args.distinct = saved
        ref_steps = max(1, min(args.steps, 20))   # each step is a bounded sample; the whole arm stays within a few minutes
        fps, cores, kind, sample = time_cpu_reference(wl, opts, args.cpu_seqs, ref_steps, min(args.warmup, 3))
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "impl": "reference", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * args.cpu_seqs / fps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "i32/f32+f64", "data": "synthetic",
            "config": dict(cfg_common, sample=f"each step = {args.cpu_seqs} of the sequences (bounded sample)"),
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return

    # ---------------- B200 arm ----------------
    if world > 1:
        # A rank's step uses four streams at once (landmark tracker + pose chain, candidate tracker, pyramid prefetch,
        # read-backs) and CUDA maps streams onto 8 hardware queues by default; NCCL's own streams shift that mapping, and two
        # of the step's streams on one queue serialise (head-of-line blocking) -- the suspected reason for the 0.08 ms per
        # step a shard loses under torchrun (DESIGN.md section 6).  One queue per stream; read by the driver at initialisation.
        os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 arm has no CPU fallback (use --impl reference for the cv2 path)")
    torch.cuda.set_device(local)
    affinity = None
    if world > 1:
        affinity = guarded(pin_to_gpu_cores, local)     # each rank on the cores (NUMA node) next to its GPU: its page-locked pool lands there
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    elif os.environ.get("B200VO_FORCE_NCCL"):   # A/B switch: a one-rank process group, to see what NCCL's presence alone costs
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
    from monocular_visual_odometry_va4mr_b200 import _lib, sharding
    ctx = _lib.Context(local)
    if n_local <= 0:
        raise SystemExit(f"bench.py: rank {rank} owns no sequence ({args.batch} sequences over {world} ranks)")
    counts = [shard_plan(args.batch, world, r, args.scaling)[1] for r in range(world)]
    wl = make_workload(args, n_local, first)
    arm = Arm(args, opts, ctx, wl, world, local, total)
    K, W = arm.K, arm.W

    clk_samples, stop = [], threading.Event()
    th = threading.Thread(target=clocks_sampler, args=(stop, clk_samples, local), daemon=True)
    if not os.environ.get("B200VO_NO_CLOCK_SAMPLER"):   # A/B switch: does the sampling thread cost the timed loop anything?
        th.start()
    res = arm.device_resident(counts)
    value = total * K / (res["dev_ms"] * 1e-3)
    e2e = guarded(arm.e2e)
    stop.set()
    if th.is_alive():
        th.join(timeout=2)
    clocks = summarize_clocks(clk_samples)

    if args.dump_outputs and rank == 0:
        dump_outputs(arm, res, args.dump_outputs)
    roofline, levels = klt_roofline(args, opts, wl, res, ROOFLINE_NOTE)
    parity = None if args.no_parity or rank != 0 else guarded(parity_check, arm, res)
    solo = rank == 0 and world == 1 and not args.no_single
    detect = guarded(measure_detect, arm) if solo else None
    arm.close()
    single = guarded(measure_single, args, opts, ctx, W) if solo else None
    bootstrap = guarded(measure_bootstrap, args) if solo else None

    # ---- extra: the other scaling form at N > 1 (at N = 1 the two coincide) ----
    other = None
    if world > 1 and not args.no_weak:
        def other_arm():
            mode = "weak" if args.scaling == "strong" else "strong"
            f2, n2, tot2 = shard_plan(args.batch, world, rank, mode)
            wl2 = make_workload(args, n2, f2)
            arm2 = Arm(args, opts, ctx, wl2, world, local, tot2)
            try:
                r2 = arm2.device_resident([shard_plan(args.batch, world, r, mode)[1] for r in range(world)])
                s2, _, _ = arm2.timed_host_loop(True)
                s2 = arm2.max_over_ranks([s2])[0]
            finally:
                arm2.close()
            return {"scaling": mode, "sequences_per_gpu": n2, "sequences_total": tot2, "value": tot2 * K / (r2["dev_ms"] * 1e-3),
                    "ms_per_step": r2["dev_ms"] / K, "e2e_value": tot2 * K / s2, "e2e_ms_per_step": 1e3 * s2 / K,
                    "what": "same measurement with the other partitioning: weak = --batch sequences on EVERY GPU, strong = --batch in total"}
        # every rank must take part (collectives inside); only rank 0 reports
        other = guarded(other_arm)

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = guarded(lambda: dict(zip(("value", "cores", "kind", "sample"),
                                           time_cpu_reference(wl, opts, args.cpu_seqs, args.cpu_steps, 2))))
            if "error" not in cpu:
                cpu = {"value": cpu["value"], "unit": "frames/s", "cores": cpu["cores"], "kind": cpu["kind"], "sample": cpu["sample"]}
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": res["dev_ms"] / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "i32/f32+f64", "data": "synthetic",
            "config": dict(cfg_common, sequences_per_gpu=counts, pyramid_levels=levels, pnp_ok_last_step=res["n_ok"],
                           distinct_scenes=args.distinct, gathered_sequences=res["gathered_sequences"],
                           device_loop=("frames of step t+1 handed over one step ahead (b200vo_batch_submit_frames_dev), consumed by "
                                        "b200vo_batch_step_dev(frames=NULL)" if not args.no_lookahead else "b200vo_batch_step_dev(frames)"),
                           parallelism=f"sequences sharded x{world} ({args.scaling} scaling), NCCL all_gather of poses"),
            "clocks": clocks,
            "cpu_affinity_cores": affinity, "cuda_device_max_connections": os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"),
            "e2e": e2e,
            "gpu_launches": res["launches"],
            "roofline": roofline,
            "cpu_baseline": cpu,
            "parity_checked": bool(parity and parity.get("ok")),
            "parity": parity,
            "single_sequence": single,
            "detect": detect,
            "bootstrap": bootstrap,
            ("weak_scaling" if args.scaling == "strong" else "strong_scaling"): other,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)
    main()
