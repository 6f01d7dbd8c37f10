"""Randomised differential run: CUDA path (through the C ABI) vs the oracle, many shapes / sizes / seeds.
Not collected by pytest (it runs for minutes); prints every mismatch.

  python tests/fuzz_parity.py [seconds]          (FUZZ_SEED=n for another stream, FUZZ_KINDS=batch for the batch kind alone)

Round-1 record: 240 s on a B200 = 632 tracker calls (random image sizes 120..900 x 90..500, six window
sizes, maxLevel 0..6, all three criteria types, points on quarter-pixel grids and with 3.2e-5 offsets),
211 goodFeaturesToTrack, 210 knnMatch (with planted duplicate descriptors), 210 solvePnPRansac,
210 findEssentialMat + recoverPose, 210 min-distance masks: 0 mismatches.  Seeds 2 and 3 (500 s, + 428
triangulation loops): one findEssentialMat mask differing in ONE point (threshold tie, see below), nothing else.
Seed 4 (330 s, 3 372 calls) and seed 6 on the final round-1 binary (300 s, 3 012 calls): 0 mismatches.
Round 2 (SIFT added; persistent tracker, fused pose kernel, second kNN kernel): seed 11 (180 s) one findEssentialMat case with
4 mask points -- an ill-conditioned sample on which cv2 sides with the CUDA path (DESIGN.md section 2 fact 5; the oracle's
root termination was aligned afterwards); seeds 21 and 22 (240 s each, 1 700 + 1 800 calls incl. 303 SIFT frames of random
sizes) and, after the last kernel changes (branch-free kNN scan, tracker queue fix), seeds 31 and 32 (3 450 calls): 0 mismatches.
Round 3 (the batch kind: SequenceBatch with per-sequence frame sizes, compared per sequence with the oracle on its own image;
random slots up to 519 x 1299, 1-8 sequences of random and near-minimal sizes, the six windows, maxLevel 0..7, all three criteria
types, zero or random padding, two tracker steps and one detection): FUZZ_KINDS=batch, seeds 41 and 42, 250 s each, run side by
side on one B200 = 496 + 467 batches, 7 600 + 7 352 per-sequence tracker comparisons, 2 222 + 2 153 per-sequence detections:
0 mismatches."""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import numpy as np  # noqa: E402

import oracle  # noqa: E402
from make_golden import make_emat_pair, make_pnp_case, sift_like  # noqa: E402
from monocular_visual_odometry_va4mr_b200 import _lib, cv2_compat, hotpath, synth  # noqa: E402
from monocular_visual_odometry_va4mr_b200.batch import SequenceBatch  # noqa: E402

WINDOWS = [(15, 15), (21, 21), (9, 13), (31, 31), (5, 7), (21, 15)]


def batch_case(rng, bad, stats):
    """SequenceBatch with per-sequence frame sizes: a random slot, random sizes (near-minimal ones included), window,
    maxLevel, criteria and padding; two tracker steps and one detection, each sequence against the oracle on its own image."""
    win = WINDOWS[int(rng.integers(0, len(WINDOWS)))]
    slot = (int(rng.integers(win[1] + 1, 520)), int(rng.integers(win[0] + 1, 1300)))
    ml = int(rng.integers(0, 8))
    crit = (int(rng.choice([1, 2, 3])), int(rng.integers(1, 40)), float(rng.choice([0.01, 0.03, 0.001])))
    b = int(rng.integers(1, 9))

    def dim(lo, hi):          # near-minimal, near-full or anywhere
        u = rng.random()
        return int(rng.integers(lo, min(lo + 4, hi) + 1)) if u < 0.3 else hi - int(rng.integers(0, 3)) if u < 0.45 else int(rng.integers(lo, hi + 1))
    sizes = [(dim(win[1] + 1, slot[0]), dim(win[0] + 1, slot[1])) for _ in range(b)]
    sizes = [(max(win[1] + 1, r), max(win[0] + 1, c)) for r, c in sizes]
    full = synth.render_sequence(str(rng.choice(["kitti", "parking", "malaga"])), 3, seed=int(rng.integers(0, 1000)),
                                 width=slot[1], height=slot[0], start=int(rng.integers(0, 5)))["frames"]
    crops = []
    for r, c in sizes:
        y0, x0 = int(rng.integers(0, slot[0] - r + 1)), int(rng.integers(0, slot[1] - c + 1))
        crops.append(np.ascontiguousarray(full[:, y0:y0 + r, x0:x0 + c]))
    random_pad = rng.random() < 0.5

    def layout(f):
        out = rng.integers(0, 256, (b,) + slot, dtype=np.uint8) if random_pad else np.zeros((b,) + slot, np.uint8)
        for k, im in enumerate(crops):
            out[k, :im.shape[1], :im.shape[2]] = im[f]
        return out

    pts = []
    for r, c in sizes:
        n = int(rng.integers(1, 600))
        p = np.column_stack([rng.uniform(-20, c + 20, n), rng.uniform(-20, r + 20, n)]).astype(np.float32)
        if rng.random() < 0.5:
            p = np.rint(p * 4) / 4
        if rng.random() < 0.3:
            p += np.float32(3.2e-5)
        pts.append(np.ascontiguousarray(p, np.float32))
    L = max(len(p) for p in pts)
    lm = np.zeros((b, L, 2), np.float32)
    for k, p in enumerate(pts):
        lm[k, :len(p)] = p
    cand = np.zeros_like(lm)
    for k, p in enumerate(pts):
        cand[k, :len(p)] = p[::-1]
    n_pts = np.int32([len(p) for p in pts])
    n_cand = np.int32([len(p) if rng.random() < 0.7 else 0 for p in pts])
    cand_of = [np.ascontiguousarray(cand[k, :n_cand[k]]) for k in range(b)]
    sb = SequenceBatch(b, *slot, synth.K_KITTI, win=win, max_level=ml, criteria=crit, max_landmarks=max(L, 4), max_candidates=L,
                       frame_size=sizes)
    obj = np.zeros((b, max(L, 4), 3), np.float32)
    lm4 = np.zeros((b, max(L, 4), 2), np.float32)
    lm4[:, :L] = lm
    sb.prime(layout(0))
    try:
        for f in (1, 2):
            out = {k: np.array(v) for k, v in sb.step(layout(f), lm4, obj, n_pts, cand, n_cand).items()}
            for k, (r, c) in enumerate(sizes):
                for name, p in (("lm", pts[k]), ("cand", cand_of[k])):
                    if not len(p):
                        continue
                    rp, rst, _ = oracle.calc_optical_flow_pyr_lk(crops[k][f - 1], crops[k][f], p, win, ml, crit)
                    st, nxt = out[name + "_status"][k, :len(p)], out[name + "_next"][k, :len(p)]
                    ok = rst.ravel() == 1
                    if not (np.array_equal(st, rst.ravel()) and np.array_equal(nxt[ok], rp[ok])):
                        bad.append(("batch-klt", slot, (r, c), win, ml, crit, f, name, int((st != rst.ravel()).sum())))
                    stats["batch_klt"] += 1
        mc = int(rng.choice([1, 7, 50, 1400, 5000]))
        q = float(rng.choice([0.1, 0.03, 0.01, 0.3]))
        md = float(rng.choice([1, 2, 3, 5, 7.5, 10, 25]))
        cell = int(np.rint(md))
        if -(-slot[0] // cell) * -(-slot[1] // cell) * 16 > 200 * 1024:
            md = float(rng.choice([10, 25]))
        try:
            corners, nc = sb.good_features(mc, q, md)
        except _lib.B200VOError as e:
            if "exceed" not in str(e):      # more candidates than the batched path ranks: refused, not wrong
                raise
            return
        for k in range(b):
            want = oracle.good_features_to_track(crops[k][2], mc, q, md)
            want = np.zeros((0, 2), np.float32) if want is None else want.reshape(-1, 2)
            if nc[k] != len(want) or not np.array_equal(corners[k, :nc[k]], want):
                bad.append(("batch-gftt", slot, sizes[k], mc, q, md, int(nc[k]), len(want)))
            stats["batch_gftt"] += 1
    finally:
        sb.close()


def main():
    budget = float(sys.argv[1]) if len(sys.argv) > 1 else 120.0
    rng = np.random.default_rng(int(os.environ.get("FUZZ_SEED", "1")))
    t_end = time.time() + budget
    stats = dict(klt=0, gftt=0, knn=0, pnp=0, emat=0, rpose=0, mind=0, tri=0, sift=0, batch=0, batch_klt=0, batch_gftt=0)
    bad = []
    # FUZZ_KINDS=batch: only the batch kind
    only_batch = os.environ.get("FUZZ_KINDS", "") == "batch"

    def rand_frames():
        shape = str(rng.choice(["kitti", "parking", "malaga"]))
        w, h = int(rng.integers(120, 900)), int(rng.integers(90, 500))
        return synth.render_sequence(shape, 2, seed=int(rng.integers(0, 1000)), width=w, height=h, start=int(rng.integers(0, 5)))

    it = 0
    while time.time() < t_end:
        it += 1
        kind = 9 if only_batch else it % 10
        try:
            if kind == 9:
                batch_case(rng, bad, stats)
                stats["batch"] += 1
            elif kind in (0, 1, 2):
                f0, f1 = rand_frames()["frames"]
                h, w = f0.shape
                win = [(15, 15), (21, 21), (9, 13), (31, 31), (5, 7), (21, 15)][int(rng.integers(0, 6))]
                if w <= win[0] + 2 or h <= win[1] + 2:
                    continue
                ml = int(rng.integers(0, 7))
                crit = (int(rng.choice([1, 2, 3])), int(rng.integers(1, 40)), float(rng.choice([0.01, 0.03, 0.001])))
                n = int(rng.integers(1, 1500))
                pts = np.column_stack([rng.uniform(-20, w + 20, n), rng.uniform(-20, h + 20, n)]).astype(np.float32)
                if rng.random() < 0.5:
                    pts = np.rint(pts * 4) / 4          # quarter-pixel grid: exact ties in floor / round
                if rng.random() < 0.3:
                    pts += np.float32(3.2e-5)           # the negative-weight corner (DESIGN.md section 2, fact 6)
                pts = np.ascontiguousarray(pts, np.float32)
                p, st, err = cv2_compat.calcOpticalFlowPyrLK(f0, f1, pts, None, winSize=win, maxLevel=ml, criteria=crit)
                rp, rst, rerr = oracle.calc_optical_flow_pyr_lk(f0, f1, pts, win, ml, crit)
                ok = rst.ravel() == 1
                if not (np.array_equal(st, rst) and np.array_equal(p[ok], rp[ok]) and np.array_equal(err[rst == 1], rerr[rst == 1])):
                    bad.append(("klt", (w, h), win, ml, crit, n, int((st != rst).sum()), float(np.abs(p - rp)[ok].max()) if ok.any() else 0))
                stats["klt"] += 1
            elif kind == 8:
                f0 = rand_frames()["frames"][0]
                a = cv2_compat.sift_detect_and_compute(f0)
                b = oracle.sift_detect_and_compute(f0)
                if not all(np.array_equal(x, y) for x, y in zip(a, b)):      # keypoints, octave codes, descriptors: bit for bit
                    bad.append(("sift", f0.shape, len(a[0]), len(b[0])))
                stats["sift"] += 1
            elif kind == 3:
                f0 = rand_frames()["frames"][0]
                mc = int(rng.choice([0, 50, 1400, 5000]))
                q = float(rng.choice([0.1, 0.03, 0.01, 0.3]))
                md = float(rng.choice([10, 3, 1, 25, 0, 7.5]))
                a = cv2_compat.goodFeaturesToTrack(f0, mc, q, md, blockSize=3)
                b = oracle.good_features_to_track(f0, mc, q, md, 3)
                if (a is None) != (b is None) or (a is not None and not np.array_equal(a, b)):
                    bad.append(("gftt", f0.shape, mc, q, md))
                stats["gftt"] += 1
            elif kind == 4:
                nq, nt = int(rng.integers(1, 3000)), int(rng.integers(2, 3000))
                q, t = sift_like(nq, int(rng.integers(0, 99))), sift_like(nt, int(rng.integers(100, 199)))
                if rng.random() < 0.5:                  # exact duplicates -> ties (lowest train index first)
                    t[rng.integers(0, nt, nt // 10)] = q[rng.integers(0, nq, nt // 10)]
                i1, d1, a1 = cv2_compat.knn2_ratio(q, t, 0.8)
                i2, d2, a2 = oracle.knn2_ratio(q, t, 0.8)
                if not (np.array_equal(i1, i2) and np.array_equal(d1, d2) and np.array_equal(a1, a2)):
                    bad.append(("knn", nq, nt))
                stats["knn"] += 1
            elif kind == 5:
                n, of = int(rng.integers(4, 3000)), float(rng.uniform(0, 0.8))
                iters, thr = int(rng.choice([100, 500, 2000])), float(rng.choice([8, 5, 2]))
                case_seed = int(rng.integers(0, 10000))
                obj, img, K = make_pnp_case(n, of, case_seed)
                ok, rv, tv, inl = cv2_compat.solvePnPRansac(obj, img, K, np.zeros(4), flags=cv2_compat.SOLVEPNP_P3P, confidence=0.99,
                                                            reprojectionError=thr, iterationsCount=iters)
                ro, rrv, rtv, rinl, _ = oracle.solve_pnp_ransac_p3p(obj, img, K, iters, thr, 0.99)
                same = ok == ro and ((not ok) or np.array_equal(inl, rinl))
                if same and ok and len(inl) >= 6:       # EPnP on < 6 points is not pinned (DESIGN.md section 2, fact 3)
                    same = np.abs(rv - rrv).max() < 1e-6 and np.abs(tv - rtv).max() < 1e-6 * max(1, np.abs(rtv).max())
                if not same:
                    bad.append(("pnp", n, of, iters, thr, "seed", case_seed))
                stats["pnp"] += 1
            elif kind == 6:
                n, of = int(rng.integers(5, 3000)), float(rng.uniform(0, 0.6))
                case_seed = int(rng.integers(0, 10000))
                p1, p2, K = make_emat_pair(n, of, case_seed)
                E, m = cv2_compat.findEssentialMat(p1, p2, K, method=cv2_compat.RANSAC, prob=0.99, threshold=1)
                Eo, mo, _ = oracle.find_essential_mat(p1, p2, K, 0.99, 1.0, 1000)
                # the CUDA five-point solver (warp-cooperative, Jacobi-style Aberth) and the oracle's (sequential) agree to
                # ~1e-13 in E on well-conditioned samples; a sample whose det B(z) has a close root cluster can give them
                # different models (DESIGN.md section 2 fact 5: ~0.1 % of the calls, cv2 itself differs as often)
                if (E is None) != (Eo is None) or (E is not None and int((m != mo).sum()) > 1):
                    bad.append(("emat", n, of, None if E is None else int((m != mo).sum()), "seed", case_seed))
                elif E is not None:
                    g1, R1, t1, k1 = cv2_compat.recoverPose(E, p1, p2, K)
                    g2, R2, t2, k2 = oracle.recover_pose(E, p1, p2, K)
                    if g1 != g2 or not np.array_equal(k1, k2) or np.abs(R1 - R2).max() > 1e-12:
                        bad.append(("rpose", n, of, g1, g2))
                    stats["rpose"] += 1
                stats["emat"] += 1
            else:
                n, m = int(rng.integers(0, 1500)), int(rng.integers(0, 3000))
                pts = np.rint(rng.uniform(0, 1200, (n, 2))).astype(np.float32)
                ex = rng.uniform(0, 1200, (m, 2)).astype(np.float32)
                if n and m:
                    k = min(n, m) // 2
                    ex[:k] = pts[:k] + np.float32([6, 8])          # distance exactly 10
                if not np.array_equal(hotpath.min_distance_mask(pts, ex, 10.0), oracle.min_distance_mask(pts, ex, 10.0)):
                    bad.append(("mind", n, m))
                stats["mind"] += 1
                # triangulation loop: random scene points seen from random past poses, random age / parallax / depth gates
                n = int(rng.integers(1, 1200))
                n_poses = int(rng.integers(1, 6))
                K = synth.K_KITTI
                transforms = []
                for j in range(n_poses):
                    R, c = synth.Corridor.pose(int(rng.integers(0, 12)), float(rng.choice([0.8, 0.15, 0.0])))
                    transforms.append((R, c.reshape(3, 1)))
                Rc, cc = synth.Corridor.pose(int(rng.integers(0, 14)), 0.8)
                Xw = np.column_stack([rng.uniform(-8, 8, n), rng.uniform(-2, 1.6, n), rng.uniform(-5, 300, n)])
                fp = rng.integers(0, n_poses, n)
                p0 = np.empty((n, 2), np.float32)
                for j in range(n_poses):
                    sel = fp == j
                    if sel.any():
                        p0[sel] = synth.project(K, transforms[j][0], transforms[j][1].ravel(), Xw[sel]).astype(np.float32)
                p1 = (synth.project(K, Rc, cc, Xw) + rng.normal(0, 0.5, (n, 2))).astype(np.float32)
                p0 = np.nan_to_num(p0, nan=0.0, posinf=1e6, neginf=-1e6).astype(np.float32)
                p1 = np.nan_to_num(p1, nan=0.0, posinf=1e6, neginf=-1e6).astype(np.float32)
                opt = dict(min_dist_landmarks=float(rng.choice([0, 1])), max_dist_landmarks=float(rng.choice([50, 100, 150])),
                           min_baseline_angle=float(rng.choice([0, 0.5, 2])), min_baseline_frames=int(rng.integers(0, 3)))
                k1, l1, q1 = hotpath.triangulate_landmarks(K, opt, p0, p1, fp, transforms, Rc, cc.reshape(3, 1))
                k2, l2, q2 = oracle.triangulate_landmarks(K, (opt["min_dist_landmarks"], opt["max_dist_landmarks"], opt["min_baseline_angle"],
                                                              opt["min_baseline_frames"]), p0, p1, fp, oracle.pack_poses(transforms),
                                                          np.hstack([Rc.reshape(9), cc.reshape(3)]))
                if not (np.array_equal(k1, k2) and np.array_equal(q1, q2) and l1.shape == l2.shape
                        # one float32 ulp of the landmark's largest coordinate (a coordinate that cancels to ~1e-15 is noise)
                        and (len(l1) == 0 or np.all(np.abs(l1 - l2) <= np.spacing(np.abs(l2).max(axis=1, keepdims=True))))):
                    bad.append(("tri", n, n_poses, int((k1 != k2).sum())))
                stats["tri"] += 1
        except Exception as e:  # noqa: BLE001
            bad.append(("EXC", kind, repr(e)[:200]))
    print("runs", stats)
    print("mismatches", len(bad))
    for b in bad[:40]:
        print(b)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
