"""The tracker's level paths against the oracle, bit for bit: template derivatives from the unrounded bilinear grid
(windows whose tap grid is inside the image) next to the per-tap path (windows at the image edges) in one launch,
the exact hi/lo iteration sums of high-contrast windows, a negative bilinear weight on the interior path, and runs
with and without the error output."""
import numpy as np
import pytest

from monocular_visual_odometry_va4mr_b200 import _lib, synth

pytestmark = pytest.mark.gpu

CRIT = (3, 30, 0.01)


@pytest.fixture(scope="module")
def env():
    import torch
    return _lib.default_context(0), torch


def _track(env, f0, f1, pts, win, ml, with_err):
    """Device-pointer entry; without the error output the tracker skips Iwin and the final error pass."""
    ctx, torch = env
    dev = torch.device("cuda", 0)
    h, w = f0.shape
    n = len(pts)
    d0, d1 = torch.from_numpy(f0).to(dev), torch.from_numpy(f1).to(dev)
    dp = torch.from_numpy(np.ascontiguousarray(pts, np.float32)).to(dev)
    o_p = torch.zeros((n, 2), dtype=torch.float32, device=dev)
    o_s = torch.zeros((n,), dtype=torch.uint8, device=dev)
    o_e = torch.zeros((n,), dtype=torch.float32, device=dev)
    rc = ctx.lib.b200vo_calc_optical_flow_pyr_lk_dev(ctx.h, d0.data_ptr(), d1.data_ptr(), h, w, w, w, dp.data_ptr(), n,
                                                     win[0], win[1], ml, CRIT[0], CRIT[1], CRIT[2], 0, 1e-4, o_p.data_ptr(),
                                                     o_s.data_ptr(), o_e.data_ptr() if with_err else 0)
    assert rc == 0, ctx.last_error()
    ctx.sync()
    torch.cuda.synchronize()
    return o_p.cpu().numpy(), o_s.cpu().numpy(), o_e.cpu().numpy()


def _check_both(env, f0, f1, pts, win, ml):
    import oracle
    rp, rst, rerr = oracle.calc_optical_flow_pyr_lk(f0, f1, pts, win, ml, CRIT)
    rst, rerr = rst.ravel(), rerr.ravel()
    ok = rst == 1
    p, st, err = _track(env, f0, f1, pts, win, ml, True)
    assert np.array_equal(st, rst)
    assert np.array_equal(p[ok], rp[ok]) and np.array_equal(err[ok], rerr[ok])
    q, st2, _ = _track(env, f0, f1, pts, win, ml, False)
    assert np.array_equal(st2, rst) and np.array_equal(q[ok], rp[ok])
    return ok


def _edge_points(w, h, win, ml, rng):
    """Points whose level-L windows straddle each image edge at every level L, plus interior points."""
    pts = []
    for lvl in range(ml + 1):
        s = 1 << lvl
        for d in range(-2, win[0] + 3):
            for _ in range(2):
                f = rng.uniform(0, 1, 2)
                pts.append(((d + f[0]) * s, rng.uniform(0.3, 0.7) * h))
                pts.append((w - 1 - (d + f[0]) * s, rng.uniform(0.3, 0.7) * h))
                pts.append((rng.uniform(0.3, 0.7) * w, (d + f[1]) * s))
                pts.append((rng.uniform(0.3, 0.7) * w, h - 1 - (d + f[1]) * s))
    pts += list(zip(rng.uniform(40, w - 40, 200), rng.uniform(40, h - 40, 200)))
    return np.float32(pts)


@pytest.mark.parametrize("win,ml", [((15, 15), 5), ((15, 15), 3), ((21, 21), 3)])
def test_edge_and_interior_windows_vs_oracle(env, win, ml):
    s = synth.render_sequence("kitti", 2, seed=11)
    f0, f1 = s["frames"]
    h, w = f0.shape
    pts = _edge_points(w, h, win, ml, np.random.default_rng(4))
    ok = _check_both(env, f0, f1, pts, win, ml)
    assert 100 < ok.sum() < len(pts)


@pytest.mark.parametrize("win", [(15, 15), (21, 21)])
def test_high_contrast_wide_sums_vs_oracle(env, win):
    """A checkerboard puts lane sums of dIx^2 far above the single-REDUX bound: the hi/lo sums run."""
    h, w = 240, 400
    yy, xx = np.mgrid[0:h, 0:w]
    board = (((xx // 6) + (yy // 6)) % 2 * 255).astype(np.float32)
    rng = np.random.default_rng(7)
    f0 = np.clip(board + rng.normal(0, 6, board.shape), 0, 255).astype(np.uint8)
    shifted = (((xx - 1.4) // 6 + (yy - 0.6) // 6) % 2 * 255).astype(np.float32)
    f1 = np.clip(shifted + rng.normal(0, 6, board.shape), 0, 255).astype(np.uint8)
    pts = np.float32(np.stack([rng.uniform(20, w - 20, 300), rng.uniform(20, h - 20, 300)], 1))
    ok = _check_both(env, f0, f1, pts, win, 2)
    assert ok.sum() > 100


@pytest.mark.parametrize("win,ml", [((15, 15), 0), ((15, 15), 3), ((21, 21), 0)])
def test_negative_bilinear_weight_interior_vs_oracle(env, win, ml):
    """iw11 = -1 (three rounded weights adding up to 2^14 + 1) at interior windows: U and its derivatives carry it."""
    s = synth.render_sequence("kitti", 2, seed=0)
    f0, f1 = s["frames"]
    sc, one = np.float32(16384), np.float32(1)
    pts = []
    for base in range(30, 340):
        x = np.float32(base)
        for _ in range(12):
            x = np.nextafter(x, np.float32(1e9))
            a = np.float32(x - np.float32(7)) - np.floor(np.float32(x - np.float32(7)))
            if 16384 - int(np.rint((one - a) * (one - a) * sc)) - 2 * int(np.rint(a * (one - a) * sc)) < 0:
                pts.append((x, x))
                break
    pts = np.ascontiguousarray(np.float32(pts))
    assert len(pts) >= 50
    ok = _check_both(env, f0, f1, pts, win, ml)
    assert ok.sum() > 10
