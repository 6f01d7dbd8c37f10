"""Seeded synthetic scenes shaped like the reference's three datasets.

The reference loads KITTI / Malaga / Parking frames from disk (reference
``utils.py:11-85``); those datasets are not available offline, so tests and the
benchmark render a procedurally textured, piecewise-planar corridor under a
known camera trajectory with the reference's real intrinsics
(``utils.py:22-24`` KITTI, ``:34-36`` Malaga, ``:43-45`` Parking).

numpy only: this module travels to the GPU box and must not need cv2.
"""
from __future__ import annotations

import numpy as np

# Intrinsics copied as *values* from the reference (utils.py:22-24, 34-36, 43-45).
K_KITTI = np.array([[718.856, 0.0, 607.1928], [0.0, 718.856, 185.2157], [0.0, 0.0, 1.0]])
K_MALAGA = np.array([[621.18428, 0.0, 404.0076], [0.0, 621.18428, 309.05989], [0.0, 0.0, 1.0]])
K_PARKING = np.array([[331.37, 0.0, 320.0], [0.0, 369.568, 240.0], [0.0, 0.0, 1.0]])

SHAPES = {
    # name: (K, width, height, forward step [m], PnP reprojection error)
    "kitti": (K_KITTI, 1241, 376, 0.8, 8.0),
    "parking": (K_PARKING, 640, 480, 0.15, 5.0),
    "malaga": (K_MALAGA, 1024, 768, 0.4, 5.0),
}

_TEX = 1024  # texture side (texels); wraps


def _value_noise(rng: np.random.Generator, size: int) -> np.ndarray:
    """Multi-octave value noise in [0,1], float32 (size x size)."""
    out = np.zeros((size, size), np.float32)
    amp_sum = 0.0
    for octave, amp in ((8, 1.0), (32, 0.8), (128, 0.6), (512, 0.45)):
        g = rng.random((octave + 1, octave + 1), dtype=np.float32)
        xs = np.linspace(0, octave, size, endpoint=False, dtype=np.float32)
        i0 = np.floor(xs).astype(np.int32)
        f = xs - i0
        f = f * f * (3 - 2 * f)
        rows = g[i0] * (1 - f)[:, None] + g[i0 + 1] * f[:, None]          # (size, octave+1)
        layer = rows[:, i0] * (1 - f)[None, :] + rows[:, i0 + 1] * f[None, :]
        out += amp * layer
        amp_sum += amp
    return out / amp_sum


def make_texture(seed: int, size: int = _TEX) -> np.ndarray:
    """Noise + random rectangles, float32 grey levels around 130 +- 35."""
    rng = np.random.default_rng(seed)
    tex = 60.0 + 140.0 * _value_noise(rng, size)
    n_rect = 900
    x0 = rng.integers(0, size, n_rect)
    y0 = rng.integers(0, size, n_rect)
    w = rng.integers(4, 40, n_rect)
    h = rng.integers(4, 40, n_rect)
    val = rng.uniform(-70.0, 70.0, n_rect).astype(np.float32)
    for i in range(n_rect):
        tex[y0[i]:y0[i] + h[i], x0[i]:x0[i] + w[i]] += val[i]
    return np.clip(tex, 0.0, 255.0).astype(np.float32)


class Corridor:
    """Ground plane y=+1.65 (camera y-down), walls x=+-6, backdrop z=z_back."""

    def __init__(self, seed: int = 0, z_back: float = 1000.0):
        self.seed = seed
        self.z_back = z_back
        self.tex = [make_texture(seed * 16 + i) for i in range(4)]

    @staticmethod
    def pose(i: int, step: float) -> tuple[np.ndarray, np.ndarray]:
        """Camera-in-world pose of frame i: (R_cw 3x3, c 3) -- forward motion, slow yaw."""
        yaw = 0.03 * np.sin(i * 0.07)
        cy, sy = np.cos(yaw), np.sin(yaw)
        R = np.array([[cy, 0.0, sy], [0.0, 1.0, 0.0], [-sy, 0.0, cy]])
        c = np.array([0.4 * np.sin(i * 0.05), 0.0, step * i])
        return R, c

    def _lookup(self, tex: np.ndarray, u: np.ndarray, v: np.ndarray) -> np.ndarray:
        n = tex.shape[0]
        u0 = np.floor(u)
        v0 = np.floor(v)
        fu = (u - u0).astype(np.float32)
        fv = (v - v0).astype(np.float32)
        iu = u0.astype(np.int64) % n
        iv = v0.astype(np.int64) % n
        iu1 = (iu + 1) % n
        iv1 = (iv + 1) % n
        top = tex[iv, iu] * (1 - fu) + tex[iv, iu1] * fu
        bot = tex[iv1, iu] * (1 - fu) + tex[iv1, iu1] * fu
        return top * (1 - fv) + bot * fv

    def render(self, K: np.ndarray, R_cw: np.ndarray, c: np.ndarray, width: int, height: int):
        """Returns (uint8 image HxW, float64 camera-frame depth HxW)."""
        xs, ys = np.meshgrid(np.arange(width, dtype=np.float64), np.arange(height, dtype=np.float64))
        dc = np.stack([(xs - K[0, 2]) / K[0, 0], (ys - K[1, 2]) / K[1, 1], np.ones_like(xs)], -1)
        d = dc @ R_cw.T
        big = 1e30
        with np.errstate(divide="ignore", invalid="ignore"):
            t_g = np.where(d[..., 1] > 1e-9, (1.65 - c[1]) / d[..., 1], big)
            t_l = np.where(d[..., 0] < -1e-9, (-6.0 - c[0]) / d[..., 0], big)
            t_r = np.where(d[..., 0] > 1e-9, (6.0 - c[0]) / d[..., 0], big)
            t_b = np.where(d[..., 2] > 1e-9, (self.z_back - c[2]) / d[..., 2], big)
        ts = np.stack([t_g, t_l, t_r, t_b], 0)
        ts = np.where(ts > 0, ts, big)
        which = np.argmin(ts, 0)
        t = np.take_along_axis(ts, which[None], 0)[0]
        p = c[None, None, :] + d * t[..., None]
        img = np.zeros((height, width), np.float32)
        scale = 24.0  # texels per metre on near planes
        for k in range(4):
            m = which == k
            if not m.any():
                continue
            if k == 0:
                u, v = p[..., 0][m] * scale, p[..., 2][m] * scale
            elif k in (1, 2):
                u, v = p[..., 2][m] * scale, p[..., 1][m] * scale
            else:
                u, v = p[..., 0][m] * 0.6, p[..., 1][m] * 0.6
            img[m] = self._lookup(self.tex[k], u, v)
        depth = t  # dc has z=1, so camera-frame depth == ray parameter
        return np.clip(np.rint(img), 0, 255).astype(np.uint8), depth


def render_sequence(shape: str = "kitti", n_frames: int = 3, seed: int = 0, start: int = 0,
                    width: int | None = None, height: int | None = None, K: np.ndarray | None = None):
    """Frames, depths and poses for a dataset-shaped sequence, seen by the dataset's camera or by ``K`` (3, 3).

    Returns dict(K, frames [n,H,W] u8, depth [n,H,W] f64, R_cw [n,3,3], c [n,3]).
    """
    K0, w, h, step, _ = SHAPES[shape]
    K = K0 if K is None else np.asarray(K, np.float64).reshape(3, 3)
    w = width or w
    h = height or h
    scene = Corridor(seed)
    frames, depths, Rs, cs = [], [], [], []
    for i in range(start, start + n_frames):
        R, c = scene.pose(i, step)
        img, dep = scene.render(K, R, c, w, h)
        frames.append(img)
        depths.append(dep)
        Rs.append(R)
        cs.append(c)
    return dict(K=K.copy(), frames=np.stack(frames), depth=np.stack(depths),
                R_cw=np.stack(Rs), c=np.stack(cs))


def backproject(K, R_cw, c, pts, depth_map):
    """World landmarks of pixel points (N,2) using the rendered depth (nearest pixel)."""
    xi = np.clip(np.rint(pts[:, 0]).astype(int), 0, depth_map.shape[1] - 1)
    yi = np.clip(np.rint(pts[:, 1]).astype(int), 0, depth_map.shape[0] - 1)
    z = depth_map[yi, xi]
    dc = np.stack([(pts[:, 0] - K[0, 2]) / K[0, 0], (pts[:, 1] - K[1, 2]) / K[1, 1], np.ones(len(pts))], -1)
    return c[None, :] + (dc * z[:, None]) @ R_cw.T


def project(K, R_cw, c, X):
    """Pixel projections (N,2) of world points under camera-in-world pose (R_cw, c)."""
    xc = (X - c[None, :]) @ R_cw
    return np.stack([K[0, 0] * xc[:, 0] / xc[:, 2] + K[0, 2], K[1, 1] * xc[:, 1] / xc[:, 2] + K[1, 2]], -1)


def grid_corners(img: np.ndarray, n: int, seed: int = 0, border: int = 12) -> np.ndarray:
    """n well-spread, textured, sub-pixel-jittered points (N,2) float32 -- a cv2-free stand-in
    for Shi-Tomasi seeding when only a point set of a given size is needed (bench inputs)."""
    rng = np.random.default_rng(seed)
    h, w = img.shape
    f = img.astype(np.float32)
    gx = np.abs(f[1:-1, 2:] - f[1:-1, :-2])
    gy = np.abs(f[2:, 1:-1] - f[:-2, 1:-1])
    score = np.minimum(gx, gy)
    score[:border, :] = 0
    score[-border:, :] = 0
    score[:, :border] = 0
    score[:, -border:] = 0
    flat = np.argsort(score.ravel())[::-1]
    cell = max(2, int(np.sqrt((h * w) / (4.0 * n))))
    taken = set()
    pts = []
    sw = score.shape[1]
    for idx in flat:
        y, x = divmod(int(idx), sw)
        key = (y // cell, x // cell)
        if key in taken:
            continue
        taken.add(key)
        pts.append((x + 1, y + 1))
        if len(pts) == n:
            break
    pts = np.asarray(pts, np.float32)
    if len(pts) < n:  # top up with jittered duplicates
        extra = pts[rng.integers(0, len(pts), n - len(pts))] + rng.uniform(-3, 3, (n - len(pts), 2)).astype(np.float32)
        pts = np.concatenate([pts, extra], 0)
    pts += rng.uniform(-0.5, 0.5, pts.shape).astype(np.float32)
    return np.ascontiguousarray(pts, np.float32)
