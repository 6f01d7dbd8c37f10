"""CPU reference of cv2 4.13's detection masks (test infrastructure), built on the unmasked oracle.

goodFeaturesToTrack(..., mask=) (featureselect.cpp), restated literally:
  * maxVal = minMaxLoc(eig, mask): the largest eigenvalue over the pixels of nonzero mask bytes, the 1-pixel border
    included (no corner can sit there, but it sets the threshold).  It may be negative: cornerMinEigenVal returns values
    down to about -3e-11 on quantised ramps.
  * eig thresholded TOZERO at (float)(maxVal * qualityLevel), dilated 3 x 3; a candidate is an interior pixel with a
    nonzero thresholded value equal to its dilation and a nonzero mask byte.  Any nonzero byte counts.
  * candidates ordered by (value desc, address desc), then the greedy minDistance selection on a grid of
    round(minDistance) cells, at most maxCorners.
SIFT detectAndCompute(img, mask) (sift.dispatch.cpp): after removeDuplicatedSorted and the firstOctave = -1 rescale,
KeyPointsFilter::runByPixelsMask drops a keypoint when mask[(int)(pt.y + 0.5f)][(int)(pt.x + 0.5f)] == 0, keeping order;
descriptors are computed for the survivors only, so they equal the unmasked ones.
"""
import numpy as np
from scipy.ndimage import maximum_filter

import oracle


def gftt_candidates(img, quality, mask=None, block_size=3):
    """-> (candidate addresses y * w + x in cv2's order, image width)"""
    eig = oracle.min_eig_map(img, block_size)
    h, w = eig.shape
    m = np.ones((h, w), bool) if mask is None else np.asarray(mask) != 0
    if not m.any():
        return np.zeros(0, np.int64), w
    max_val = float(eig[m].max())                                  # signed, double, as minMaxLoc returns it
    thr = np.float32(max_val * quality)
    t = np.where(eig > thr, eig, np.float32(0)).astype(np.float32)
    dil = maximum_filter(t, size=3, mode="nearest")
    c = (t != 0) & (t == dil) & m
    c[0, :] = c[-1, :] = c[:, 0] = c[:, -1] = False
    idx = np.flatnonzero(c).astype(np.int64)
    vals = eig.ravel()[idx]
    order = np.lexsort((-idx, -vals))                              # value desc, then address desc
    return idx[order], w


def good_features_to_track(img, max_corners, quality, min_dist, mask=None, block_size=3):
    """-> float32 (M, 1, 2) or None, as cv2.goodFeaturesToTrack(img, ..., mask=mask) returns them"""
    idx, w = gftt_candidates(img, quality, mask, block_size)
    h = img.shape[0]
    out = []
    if min_dist >= 1:
        cell = int(np.rint(min_dist))
        gw, gh = (w + cell - 1) // cell, (h + cell - 1) // cell
        md2 = min_dist * min_dist
        grid = {}
        for a in idx.tolist():
            y, x = divmod(a, w)
            xc, yc = x // cell, y // cell
            good = True
            for yy in range(max(0, yc - 1), min(gh - 1, yc + 1) + 1):
                for xx in range(max(0, xc - 1), min(gw - 1, xc + 1) + 1):
                    for px, py in grid.get((xx, yy), ()):
                        if (x - px) ** 2 + (y - py) ** 2 < md2:
                            good = False
                            break
                    if not good:
                        break
                if not good:
                    break
            if good:
                grid.setdefault((xc, yc), []).append((x, y))
                out.append((x, y))
                if max_corners > 0 and len(out) == max_corners:
                    break
    else:
        for a in idx.tolist()[:max_corners if max_corners > 0 else None]:
            y, x = divmod(a, w)
            out.append((x, y))
    return np.float32(out).reshape(-1, 1, 2) if out else None


def sift_mask_keep(xy, mask):
    """bool (n,): the keypoints (halved coordinates, float32) that runByPixelsMask keeps"""
    xy = np.asarray(xy, np.float32).reshape(-1, 2)
    col = (xy[:, 0] + np.float32(0.5)).astype(np.int64)           # (int) of a non-negative float32 sum
    row = (xy[:, 1] + np.float32(0.5)).astype(np.int64)
    return np.asarray(mask)[row, col] != 0


def sift_detect_and_compute(img, mask=None, max_kp=20000):
    """-> (kps float32 (n, 5), octave int32 (n,), descriptors float32 (n, 128)) of cv2's detectAndCompute(img, mask)"""
    kp, octv, desc = oracle.sift_detect_and_compute(img, max_kp)
    if mask is None:
        return kp, octv, desc
    keep = sift_mask_keep(kp[:, :2], mask)
    return kp[keep], octv[keep], desc[keep]


# ---------------------------------------------------------------- the masks the tests use
def hood_mask(shape, frac=0.2):
    """a dash camera's hood: the bottom `frac` of the rows, with rounded shoulders"""
    h, w = shape
    m = np.full(shape, 255, np.uint8)
    top = int(h * (1 - frac))
    yy, xx = np.mgrid[:h, :w]
    m[(yy >= top) & (np.abs(xx - w / 2) <= w / 2 - (yy - top) * 0.5 + w * 0.1)] = 0
    m[yy >= top + (h - top) // 2] = 0
    return m


def wedge_mask(shape, depth=0.25):
    """the black corner wedges of an undistorted image: four triangles"""
    h, w = shape
    yy, xx = np.mgrid[:h, :w].astype(np.float64)
    u, v = xx / (w - 1), yy / (h - 1)
    d = depth
    bad = (u + v < d) | ((1 - u) + v < d) | (u + (1 - v) < d) | ((1 - u) + (1 - v) < d)
    return np.where(bad, 0, 255).astype(np.uint8)


def blob_mask(shape, seed=0, n=12):
    """random discs (logos, timestamps, dirt) masked out, the rest masked in with assorted nonzero values"""
    rng = np.random.default_rng(seed)
    h, w = shape
    m = rng.integers(1, 256, shape).astype(np.uint8)
    yy, xx = np.mgrid[:h, :w]
    for _ in range(n):
        cy, cx, r = rng.integers(0, h), rng.integers(0, w), rng.integers(5, max(6, min(h, w) // 6))
        m[(yy - cy) ** 2 + (xx - cx) ** 2 <= r * r] = 0
    return m


def quiet_patch(eig, size=40):
    """(y0, x0) of the size x size interior window with the smallest maximum eigenvalue"""
    h, w = eig.shape
    best = None
    for y0 in range(8, h - size - 8, size // 2):
        for x0 in range(8, w - size - 8, size // 2):
            v = eig[y0:y0 + size, x0:x0 + size].max()
            if best is None or v < best[0]:
                best = (v, y0, x0)
    return best[1], best[2]


def patch_masks(img, size=40):
    """name -> mask: a quiet patch alone, and the same patch plus the 1-pixel border ring"""
    eig = oracle.min_eig_map(img)
    y0, x0 = quiet_patch(eig, size)
    patch = np.zeros(img.shape, np.uint8)
    patch[y0:y0 + size, x0:x0 + size] = 255
    ring = patch.copy()
    ring[0, :] = ring[-1, :] = ring[:, 0] = ring[:, -1] = 9
    return {"quiet_patch": patch, "patch_and_ring": ring}


def standard_masks(img, seed=0):
    """name -> mask of the image's shape: every mask the masked-detection tests run"""
    shape = img.shape
    out = {"hood": hood_mask(shape), "wedges": wedge_mask(shape), "blobs": blob_mask(shape, seed),
           "all_255": np.full(shape, 255, np.uint8), "all_1": np.full(shape, 1, np.uint8), "all_7": np.full(shape, 7, np.uint8),
           "all_0": np.zeros(shape, np.uint8)}
    out.update(patch_masks(img))
    return out


def ramp_images(n=200, seed=1, shape=(64, 96)):
    """quantised intensity ramps, on which cornerMinEigenVal has negative values"""
    rng = np.random.default_rng(seed)
    h, w = shape
    yy, xx = np.mgrid[:h, :w]
    for _ in range(n):
        a = rng.uniform(0, np.pi)
        yield ((np.cos(a) * xx + np.sin(a) * yy) * rng.uniform(0.5, 4)).astype(np.int64).clip(0, 255).astype(np.uint8)


def negative_eig_cases(limit=6):
    """[(image, one-pixel mask, 3 x 3 mask)] on interior pixels whose eigenvalue, and whose 3 x 3 neighbourhood's, is < 0"""
    out = []
    for img in ramp_images():
        eig = oracle.min_eig_map(img)
        h, w = eig.shape
        for y, x in np.argwhere(eig < 0):
            if 2 <= y < h - 2 and 2 <= x < w - 2 and (eig[y - 1:y + 2, x - 1:x + 2] < 0).all():
                one = np.zeros(img.shape, np.uint8)
                one[y, x] = 255
                nine = np.zeros(img.shape, np.uint8)
                nine[y - 1:y + 2, x - 1:x + 2] = 255
                out.append((img, one, nine))
                break
        if len(out) == limit:
            break
    return out


def checkerboard():
    """a checkerboard of 2 x 2 squares: plateaus of tied maxima, about 117000 candidates (the detector's sort path for
    more than 32768)"""
    yy, xx = np.mgrid[:300, :400]
    return (((yy // 2 + xx // 2) % 2) * 255).astype(np.uint8)
