#!/usr/bin/env python
"""Secondary workloads of BASELINE.json (configs 2-4): per call-site timings through the C-ABI
(host buffers in, host buffers out) next to the same cv2 call on the host cores.

  python benchmarks/bench_components.py [--only knn,gftt,klt,pnp,emat,next,sift] [--reps 20]

Prints one JSON object per workload.  `gpu_ms` is CUDA-event time on the ctx stream for the whole
call (H2D + kernels + D2H), `wall_ms` the median wall clock of the call, `cv2_ms` the median wall
clock of the cv2 call on all host threads.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def med(f, reps, warm=3):
    for _ in range(warm):
        f()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="knn,gftt,klt,pnp,emat,next,sift")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--no-cv2", action="store_true")
    args = ap.parse_args()
    only = set(args.only.split(","))
    from monocular_visual_odometry_va4mr_b200 import _lib, cv2_compat, synth
    from make_golden import make_emat_pair, make_pnp_case, sift_like
    cv2 = None
    if not args.no_cv2:
        try:
            import cv2
            cv2.setNumThreads(os.cpu_count() or 1)
        except ImportError:
            cv2 = None
    ctx = _lib.default_context(0)

    if "knn" in only:   # config 3: 8192 x 8192 x 128
        q, t = sift_like(8192, 1), sift_like(8192, 2)
        wall = med(lambda: cv2_compat.knn2_ratio(q, t, 0.8), args.reps)
        gpu = ctx.last_gpu_ms()
        r = {"workload": "knn2+ratio 8192x8192x128 (config 3)", "wall_ms": wall, "gpu_ms": gpu, "gflop": 2 * 8192 * 8192 * 128 / 1e9}
        if cv2 is not None:
            bf = cv2.BFMatcher()
            r["cv2_ms"] = med(lambda: [m for m, n in bf.knnMatch(q, t, k=2) if m.distance < 0.8 * n.distance], 3, 1)
        # page-locked caller buffers (b200vo_host_alloc): DMA'd in place, no staging copies
        import ctypes as C

        def pinned(shape, dtype):
            nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
            ptr = ctx.lib.b200vo_host_alloc(ctx.h, nbytes)
            return np.frombuffer((C.c_uint8 * nbytes).from_address(ptr), dtype).reshape(shape), ptr
        (pq, p0), (pt, p1) = pinned(q.shape, np.float32), pinned(t.shape, np.float32)
        (pi, p2), (pd, p3), (pa, p4) = pinned((8192, 2), np.int32), pinned((8192, 2), np.float32), pinned((8192,), np.uint8)
        pq[:] = q; pt[:] = t
        call = lambda: ctx.lib.b200vo_knn2_ratio(ctx.h, pq.ctypes.data_as(_lib.c_f32p), 8192, pt.ctypes.data_as(_lib.c_f32p), 8192, 128, 0.8,
                                                 pi.ctypes.data_as(_lib.c_i32p), pd.ctypes.data_as(_lib.c_f32p), pa.ctypes.data_as(_lib.c_u8p))
        r["wall_ms_pinned"] = med(call, args.reps)
        r["gpu_ms_pinned"] = ctx.last_gpu_ms()
        r["h2d_mb"] = (q.nbytes + t.nbytes) / 1e6
        # device-resident form: prep + GEMM/top-2 + finalize only
        import torch
        dev = torch.device("cuda", 0)
        dq, dt = torch.from_numpy(q).to(dev), torch.from_numpy(t).to(dev)
        oi = torch.zeros((8192, 2), dtype=torch.int32, device=dev); od = torch.zeros((8192, 2), dtype=torch.float32, device=dev)
        oa = torch.zeros((8192,), dtype=torch.uint8, device=dev)
        st = torch.cuda.ExternalStream(ctx.stream(), device=dev)
        devcall = lambda: ctx.lib.b200vo_knn2_ratio_dev(ctx.h, dq.data_ptr(), 8192, dt.data_ptr(), 8192, 128, 0.8, oi.data_ptr(), od.data_ptr(),
                                                        oa.data_ptr(), None)
        for _ in range(3):
            devcall()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(args.reps):
            devcall()
        e1.record(st)
        ctx.sync()
        r["dev_call_ms"] = e0.elapsed_time(e1) / args.reps
        r["dev_call_what"] = "b200vo_knn2_ratio_dev: f32->f16 prep x2, tcgen05 GEMM + top-2, finalize (CUDA events, back to back)"
        assert np.array_equal(oi.cpu().numpy(), pi) and np.array_equal(oa.cpu().numpy(), pa)
        for ptr in (p0, p1, p2, p3, p4):
            ctx.lib.b200vo_host_free(ctx.h, ptr)
        print(json.dumps(r))
    if "sift" in only:      # SURVEY 8f row f4: the bootstrap's detectAndCompute (reference :226-227)
        for shape in ("kitti", "parking", "malaga"):
            f = synth.render_sequence(shape, 1, seed=0)["frames"][0]
            kp, octv, des = cv2_compat.sift_detect_and_compute(f)
            wall = med(lambda: cv2_compat.sift_detect_and_compute(f), args.reps)
            r = {"workload": f"SIFT detectAndCompute {f.shape[1]}x{f.shape[0]} ({shape}-shaped)", "keypoints": int(len(kp)), "wall_ms": wall,
                 "gpu_ms": ctx.last_gpu_ms()}
            if cv2 is not None:
                sift = cv2.SIFT_create()
                r["cv2_ms"] = med(lambda: sift.detectAndCompute(f, None), 5, 1)
                r["cv2_keypoints"] = len(sift.detectAndCompute(f, None)[0])
            print(json.dumps(r))
    if "gftt" in only:
        f = synth.render_sequence("kitti", 1, seed=0)["frames"][0]
        wall = med(lambda: cv2_compat.goodFeaturesToTrack(f, 1400, 0.1, 10, blockSize=3), args.reps)
        r = {"workload": "goodFeaturesToTrack 1241x376 (1400, 0.1, 10)", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
        if cv2 is not None:
            r["cv2_ms"] = med(lambda: cv2.goodFeaturesToTrack(f, 1400, 0.1, 10, blockSize=3), args.reps)
        print(json.dumps(r))
    if "klt" in only:   # config 4 tracker part: 20k points, 21x21, 4 levels
        s = synth.render_sequence("kitti", 2, seed=0)
        f0, f1 = s["frames"]
        pts = synth.grid_corners(f0, 20000, seed=0)
        kw = dict(winSize=(21, 21), maxLevel=3, criteria=(3, 30, 0.01))
        wall = med(lambda: cv2_compat.calcOpticalFlowPyrLK(f0, f1, pts, None, **kw), args.reps)
        r = {"workload": "calcOpticalFlowPyrLK 1241x376, 20k points, 21x21, maxLevel 3 (config 4)", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
        if cv2 is not None:
            r["cv2_ms"] = med(lambda: cv2.calcOpticalFlowPyrLK(f0, f1, pts, None, **kw), 5, 1)
        print(json.dumps(r))
        pts2 = pts[:2000]
        wall = med(lambda: cv2_compat.calcOpticalFlowPyrLK(f0, f1, pts2, None, **kw), args.reps)
        r = {"workload": "calcOpticalFlowPyrLK 1241x376, 2k points, 21x21, maxLevel 3 (single call, stateless)", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
        if cv2 is not None:
            r["cv2_ms"] = med(lambda: cv2.calcOpticalFlowPyrLK(f0, f1, pts2, None, **kw), args.reps)
        print(json.dumps(r))
    if "pnp" in only:   # config 4 pose part: 20k correspondences, 2000 hypotheses
        for n, of, iters in ((20000, 0.3, 2000), (20000, 0.5, 2000), (2000, 0.1, 500)):
            obj, img, K = make_pnp_case(n, of, 4)
            kw = dict(flags=2, confidence=0.99, reprojectionError=8.0, iterationsCount=iters)
            wall = med(lambda: cv2_compat.solvePnPRansac(obj, img, K, np.zeros(4), **kw), args.reps)
            r = {"workload": f"solvePnPRansac P3P N={n} outliers={of} iters<={iters}", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
            if cv2 is not None:
                r["cv2_ms"] = med(lambda: cv2.solvePnPRansac(obj, img, K, np.zeros(4), **kw), 5, 1)
            print(json.dumps(r))
    if "emat" in only:   # bootstrap pose (config 3 tail): findEssentialMat(RANSAC, prob=0.99, threshold=1) as :308
        for n, of in ((2500, 0.2), (3000, 0.4), (500, 0.6)):
            p1, p2, K = make_emat_pair(n, of, 11)
            wall = med(lambda: cv2_compat.findEssentialMat(p1, p2, K, method=cv2_compat.RANSAC, prob=0.99, threshold=1), args.reps)
            r = {"workload": f"findEssentialMat RANSAC N={n} outliers={of}", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
            if cv2 is not None:
                r["cv2_ms"] = med(lambda: cv2.findEssentialMat(p1, p2, K, method=cv2.RANSAC, prob=0.99, threshold=1), 5, 1)
            print(json.dumps(r))
            E, _ = cv2_compat.findEssentialMat(p1, p2, K, method=cv2_compat.RANSAC, prob=0.99, threshold=1)
            wall = med(lambda: cv2_compat.recoverPose(E, p1, p2, K), args.reps)
            r = {"workload": f"recoverPose N={n} (ref :315)", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
            if cv2 is not None:
                r["cv2_ms"] = med(lambda: cv2.recoverPose(E, p1, p2, K), 5, 1)
            print(json.dumps(r))
    if "next" in only:   # SURVEY 8f: candidate min-distance filter (:258) and triangulate_landmarks (:107-206)
        from monocular_visual_odometry_va4mr_b200 import hotpath
        rng = np.random.default_rng(3)
        pts = np.rint(rng.uniform(0, 1241, (1400, 2))).astype(np.float32)
        ex = (rng.uniform(0, 1, (1500, 2)) * [1241, 376]).astype(np.float32)
        wall = med(lambda: hotpath.min_distance_mask(pts, ex, 10.0), args.reps)
        r = {"workload": "candidate min-distance filter, 1400 corners x 1500 candidates (ref :258)", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
        # the reference's own numpy expression, timed as the reference runs it (one Python iteration per corner)
        r["numpy_ms"] = med(lambda: np.array([np.all(np.linalg.norm(pts[i, :] - ex, axis=1) > 10) for i in range(pts.shape[0])]), 3, 1)
        print(json.dumps(r))
        K = synth.K_KITTI
        n = 1500
        Xw = np.column_stack([rng.uniform(-8, 8, n), rng.uniform(-2, 1.6, n), rng.uniform(5, 120, n)])
        R1, c1 = synth.Corridor.pose(3, 0.8)
        p0 = synth.project(K, np.eye(3), np.zeros(3), Xw).astype(np.float32)
        p1 = (synth.project(K, R1, c1, Xw) + rng.normal(0, 0.3, (n, 2))).astype(np.float32)
        transforms = [(np.eye(3), np.zeros((3, 1))), (np.eye(3), np.zeros((3, 1))), (np.eye(3), np.zeros((3, 1)))]
        opt = dict(min_dist_landmarks=1, max_dist_landmarks=150, min_baseline_angle=2, min_baseline_frames=2)
        fp = np.zeros(n)
        wall = med(lambda: hotpath.triangulate_landmarks(K, opt, p0, p1, fp, transforms, R1, c1.reshape(3, 1)), args.reps)
        r = {"workload": f"triangulate_landmarks candidate loop, {n} candidates (ref :170-204)", "wall_ms": wall, "gpu_ms": ctx.last_gpu_ms()}
        if cv2 is not None:   # what the reference does per candidate: one cv2.triangulatePoints call + numpy gates
            P0 = K @ np.hstack([np.eye(3), np.zeros((3, 1))])
            P1 = K @ np.hstack([R1.T, (-R1.T @ c1).reshape(3, 1)])

            def ref_loop():
                out = []
                for i in range(n):
                    X = cv2.triangulatePoints(P0, P1, p0[i].reshape(-1, 1), p1[i].reshape(-1, 1))
                    out.append(X[:3] / X[3])
                return out
            r["cv2_loop_ms"] = med(ref_loop, 3, 1)
            r["note"] = "cv2_loop_ms covers only the per-candidate cv2.triangulatePoints calls of the reference's loop (no angle/depth gates)"
        print(json.dumps(r))


if __name__ == "__main__":
    main()
