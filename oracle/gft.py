"""Oracle for Shi-Tomasi detection (sos_corner_min_eigenval / sos_gft_detect, csrc/gft.cu). TEST INFRASTRUCTURE ONLY — see
oracle/__init__.py.  NumPy only: cv2 is what the tests compare this module with, never part of its arithmetic.

  * `corner_min_eigenval` restates gft_eig_kernel operation by operation, i.e. cv2.cornerMinEigenVal(gray, 3, ksize=3):
    BORDER_REFLECT_101; Sobel in float32 with the scale s = 1 / (4 * 3 * 255) folded into the smoothing taps,
    dx = fma(s, d[-1] + d[+1], 2s * d[0]) down the column of row differences and, for dy, each row smoothed in tap order
    fma(s, g[x+1], fma(2s, g[x], s * g[x-1])) (cv2's row filter) before the difference of the rows below and above;
    products dx^2, dx dy, dy^2 in float32; 3 x 3 box sums in float64 as ((p[-1] + p[0]) + p[+1]) along the row, then the
    same down the column, rounded to float32 once; min eigenvalue (a + c) - sqrt((a - c)^2 + b^2) with a, c halved, every
    operation rounded on its own (no contraction).
  * `good_features` restates cv2.goodFeaturesToTrack (useHarrisDetector = False) on a given corner measure: threshold at
    float32(max over the mask * quality) with THRESH_TOZERO, 3 x 3 dilation, candidates = interior pixels with
    v != 0 and v == dilated and inside the mask, sorted by (value desc, pixel index desc) (cv2's greaterThanPtr), then the
    strongest-first greedy that drops a candidate closer than minDistance (dx^2 + dy^2 < minDistance^2) to an accepted
    corner; minDistance < 1 takes the list as sorted, max_corners <= 0 means no limit."""
from __future__ import annotations

import numpy as np

f32, f64 = np.float32, np.float64
SCALE = f32(1.0 / (4.0 * 3.0 * 255.0))


def refl(p, n: int):
    """BORDER_REFLECT_101 index for any n >= 1, reflected until it lands (as the kernel's refl: for n = 2 an offset of
    -2 or +2 needs two reflections)."""
    p = np.asarray(p)
    if n == 1:
        return np.zeros_like(p)
    while True:
        q = np.where(p < 0, -p, np.where(p >= n, 2 * n - 2 - p, p))
        if np.array_equal(q, p):
            return q
        p = q


def fma32(a, b, c):
    """float32 fma(a, b, c) with a single rounding, emulated in float64.  a * b is exact in float64 when the two significands
    have at most 53 bits together (here: s or 2s times an integer |k| <= 1020, at most 34 bits); the sum with c must be
    exact too, so that rounding it to float32 is the only rounding.  Both are checked, not assumed."""
    a = np.asarray(a, f32).astype(f64)
    b = np.asarray(b, f32).astype(f64)
    c = np.asarray(c, f32).astype(f64)
    p = a * b
    # Dekker: a * b is exact iff the low part of the product is zero; split each factor into 26 + 27 bits
    split = lambda v: (v * 134217729.0 - (v * 134217729.0 - v))
    ah, bh = split(a), split(b)
    al, bl = a - ah, b - bh
    err_p = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    assert not np.any(err_p), "fma32: product not exact in float64"
    s = p + c
    bb = s - p                                  # Knuth's TwoSum
    err_s = (p - (s - bb)) + (c - bb)
    assert not np.any(err_s), "fma32: sum not exact in float64"
    return s.astype(f32)


def sobel(gray: np.ndarray):
    """(dx, dy) float32 [H, W] of gft_eig_kernel: cv2.Sobel(gray, CV_32F, 1, 0 / 0, 1, ksize=3, scale=s, BORDER_REFLECT_101)."""
    g = np.asarray(gray, np.uint8)
    H, W = g.shape
    G = g.astype(f32)
    ys, xs = np.arange(H), np.arange(W)
    at = lambda dy, dx: G[refl(ys + dy, H)][:, refl(xs + dx, W)]
    s, s2 = SCALE, f32(2) * SCALE
    # rows are differentiated exactly ([-1 0 1] on integers), then smoothed down the column with (s, 2s, s)
    du, d0, dd = (at(r, 1) - at(r, -1) for r in (-1, 0, 1))
    dx = fma32(s, du + dd, (s2 * d0).astype(f32))
    # rows smoothed with (s, 2s, s) in tap order, then differenced down the column
    smooth = lambda r: fma32(s, at(r, 1), fma32(s2, at(r, 0), (s * at(r, -1)).astype(f32)))
    dy = (smooth(1) - smooth(-1)).astype(f32)
    return dx, dy


def corner_min_eigenval(gray: np.ndarray) -> np.ndarray:
    """gray uint8 [H, W] (or [n, H, W]) -> float32 corner measure of the same shape (see the module docstring)."""
    g = np.asarray(gray, np.uint8)
    if g.ndim == 3:
        return np.stack([corner_min_eigenval(x) for x in g])
    H, W = g.shape
    ys, xs = np.arange(H), np.arange(W)
    dx, dy = sobel(g)
    box = []
    for p in ((dx * dx).astype(f32), (dx * dy).astype(f32), (dy * dy).astype(f32)):
        p = p.astype(f64)
        r = (p[:, refl(xs - 1, W)] + p) + p[:, refl(xs + 1, W)]
        box.append(((r[refl(ys - 1, H)] + r) + r[refl(ys + 1, H)]).astype(f32))
    a = (box[0] * f32(0.5)).astype(f32)
    b = box[1]
    c = (box[2] * f32(0.5)).astype(f32)
    t = (a - c).astype(f32)
    r = np.sqrt(((t * t).astype(f32) + (b * b).astype(f32)).astype(f32)).astype(f32)
    return ((a + c).astype(f32) - r).astype(f32)


def candidates(eig: np.ndarray, mask, quality: float):
    """Pixel indices of the candidates of one (image, mask), sorted strongest first (value desc, index desc)."""
    eig = np.asarray(eig, f32)
    H, W = eig.shape
    m = np.ones((H, W), bool) if mask is None else np.asarray(mask).astype(bool)
    mx = f64(eig[m].max()) if m.any() else 0.0            # cv2.minMaxLoc over the mask (0 for an empty mask)
    thr = f32(mx * float(quality))
    e = np.where(eig > thr, eig, f32(0))
    pad = np.pad(e, 1, constant_values=-np.inf)
    dil = np.max([pad[1 + j:1 + j + H, 1 + i:1 + i + W] for j in (-1, 0, 1) for i in (-1, 0, 1)], axis=0)
    cand = np.zeros((H, W), bool)
    cand[1:H - 1, 1:W - 1] = True
    cand &= (e != 0) & (e == dil) & m
    idx = np.flatnonzero(cand)
    v = eig.ravel()[idx]
    return idx[np.lexsort((-idx, -v))]


def good_features(eig: np.ndarray, mask, max_corners: int, quality: float = 0.01, min_distance: float = 5.0):
    """cv2.goodFeaturesToTrack on the corner measure `eig` -> (xy float32 [k, 2] strongest first, number of candidates)."""
    H, W = np.shape(eig)
    idx = candidates(eig, mask, quality)
    ys, xs = idx // W, idx % W
    limit = len(idx) if max_corners <= 0 else int(max_corners)
    if min_distance >= 1:
        acc = np.zeros((H, W), bool)
        r, d2 = int(np.ceil(min_distance)), float(min_distance) ** 2
        out = []
        for y, x in zip(ys, xs):
            if len(out) == limit:
                break
            y0, x0 = max(0, y - r), max(0, x - r)
            yy, xx = np.nonzero(acc[y0:y + r + 1, x0:x + r + 1])
            if np.any((yy + y0 - y) ** 2 + (xx + x0 - x) ** 2 < d2):
                continue
            acc[y, x] = True
            out.append((x, y))
    else:
        out = list(zip(xs[:limit], ys[:limit]))
    return np.array(out, np.float32).reshape(-1, 2), len(idx)
