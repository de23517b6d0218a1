"""Adversarial RANSAC scoring problems for the score engines (csrc/score_mma.cuh, csrc/ransac.cu::score_kernel), shared by the
CPU model test (tests/test_score_split_cpu.py) and the GPU stress test (tests/test_gpu_score_stress.py).

Every problem has exact correspondences (sigma = 0) and an inlier fraction >= 0.7, so that most hypotheses are drawn from
all-inlier triples: good hypotheses are the ones that see pairs near the threshold.  A family fixes the geometry:

  large_motion  rotations up to 180 degrees and |t| from 0.01 to 50 x |p|
  far           |p| up to 1e3
  near_centre   a quarter of the points within 1e-3 .. 1e-1 of the current camera centre (x -> 0 in the score)
  perp_opposite bearings perpendicular (s ~ 0) and opposite (s < 0) to x; the Euclidean score gets q = -x instead
  near_thr      a quarter of the pairs planted within 1e-6 relative of the threshold (as near as float32 allows)

`scaled` multiplies every length (1000: millimetres).  With `exact_scale` the coordinates are rounded to 17 significant bits,
so that the scaled float32 inputs are exactly 1000 times the metre ones and the float64 decisions of both versions agree."""
from __future__ import annotations

import numpy as np

FAMILIES = ("large_motion", "far", "near_centre", "perp_opposite", "near_thr")
THR_BEARING = 1.0 - np.cos(np.deg2rad(5.0))
THR_EUCLID = 0.05


def rotation(rng, max_deg):
    ax = rng.normal(size=3)
    ax /= np.linalg.norm(ax)
    a = np.deg2rad(rng.uniform(-max_deg, max_deg))
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def rig_pair(rng):
    """Two cameras 0.12 m apart along z, the second one tilted by up to 10 degrees (row-major 3x4 [Rc|tc] each)."""
    Rc = rotation(rng, 10.0)
    return np.stack([np.hstack([np.eye(3), [[0.0], [0.0], [0.12]]]), np.hstack([Rc, [[0.01], [-0.02], [0.0]]])])


def round_bits(x, bits=17):
    """x rounded to `bits` significant bits (so that x * 1000 is exact in float32)."""
    m, e = np.frexp(np.asarray(x, np.float64))
    return np.ldexp(np.round(m * 2.0 ** bits) / 2.0 ** bits, e)


def unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def perpendicular(rng, u):
    w = np.cross(u, rng.normal(size=u.shape))
    return unit(w)


def tilt(rng, u, ang):
    """u rotated by `ang` (radians, per row) about a random axis perpendicular to it."""
    ax = perpendicular(rng, u)
    return u * np.cos(ang)[:, None] + np.cross(ax, u) * np.sin(ang)[:, None]


def make(rng, family, n, mode, rig=None, inlier_frac=0.75, exact_scale=False):
    """One problem in metres: (p_ref, p_cur, f_cur, cam) float32 [n,3] x3 and uint8 [n].  mode: "bearing" or "euclid".
    p_ref = R p_cur + t for inliers; the bearing of correspondence j is the direction of p_cur in its camera."""
    large = family == "large_motion"
    R = rotation(rng, 180.0 if large else 20.0)
    p_cur = unit(rng.normal(size=(n, 3)))
    if family == "far":
        p_cur *= rng.uniform(50.0, 1000.0, (n, 1))
    else:
        p_cur *= rng.uniform(0.5, 7.0, (n, 1))
    cam = np.sort((rng.random(n) < 0.5).astype(np.uint8)) if rig is not None else np.zeros(n, np.uint8)
    if family == "near_centre":   # around the centre of the point's own camera
        k = n // 4
        centre = np.asarray(rig).reshape(-1, 3, 4)[cam[:k], :, 3] if rig is not None else 0.0
        p_cur[:k] = centre + unit(p_cur[:k]) * 10.0 ** rng.uniform(-3, -1, (k, 1))
    if large:
        t = unit(rng.normal(size=3)) * np.median(np.linalg.norm(p_cur, axis=1)) * 10.0 ** rng.uniform(-2, np.log10(50.0))
    else:
        t = rng.normal(size=3) * 0.3
    p_ref = p_cur @ R.T + t
    out = rng.random(n) > inlier_frac
    scale_out = np.median(np.linalg.norm(p_ref, axis=1))
    p_ref[out] += rng.normal(size=(int(out.sum()), 3)) * scale_out * 0.3
    if exact_scale:
        p_cur = round_bits(p_cur)
    p_cur = p_cur.astype(np.float32).astype(np.float64)
    p_ref = p_ref.astype(np.float32).astype(np.float64)
    if rig is None:
        x = p_cur
    else:
        r = np.asarray(rig).reshape(-1, 3, 4)
        x = np.einsum("nji,nj->ni", r[cam, :, :3], p_cur - r[cam, :, 3])
    f = unit(x)
    inl = np.nonzero(~out)[0]
    if family == "perp_opposite":
        k = len(inl) // 8
        if mode == "bearing":
            f[inl[:k]] = perpendicular(rng, f[inl[:k]])
            f[inl[k:2 * k]] = -f[inl[k:2 * k]]
        else:
            p_ref[inl[:k]] = (-(p_cur[inl[:k]] @ R.T) + t).astype(np.float32)   # q on the far side of the camera centre
    if family == "near_thr":
        k = len(inl) // 3
        j = inl[:k]
        if mode == "bearing":
            ang = np.arccos(1.0 - THR_BEARING) * (1.0 + rng.uniform(-1e-6, 1e-6, k))
            f[j] = tilt(rng, f[j], ang)
        else:
            d = unit(rng.normal(size=(k, 3))) * THR_EUCLID * (1.0 + rng.uniform(-1e-6, 1e-6, (k, 1)))
            q = p_cur[j] @ R.T + t + d
            p_ref[j] = q.astype(np.float32)
    if exact_scale:
        p_ref = round_bits(p_ref)
    f32 = lambda a: np.ascontiguousarray(a, np.float32)
    return f32(p_ref), f32(p_cur), f32(f), cam


def scaled(prob, scale):
    """The same problem with every length multiplied by `scale` (bearings unchanged)."""
    p_ref, p_cur, f, cam = prob
    return (p_ref.astype(np.float64) * scale).astype(np.float32), (p_cur.astype(np.float64) * scale).astype(np.float32), f, cam


def scaled_rig(rig, scale):
    if rig is None:
        return None
    r = np.array(rig, np.float64).reshape(-1, 3, 4)
    r[:, :, 3] *= scale
    return r


def pose_features(M, rig):
    """Per camera (A, b) of x = A p + b for a [3,4] pose M (p_ref ~ R p_cur + t): A = Rc^T R^T, b = -Rc^T (R^T t + tc)."""
    R, t = M[:, :3], M[:, 3]
    r = np.asarray(rig, np.float64).reshape(-1, 3, 4) if rig is not None else np.hstack([np.eye(3), np.zeros((3, 1))])[None]
    A = np.einsum("cji,kj->cik", r[:, :, :3], R)                  # Rc^T R^T
    b = -np.einsum("cji,cj->ci", r[:, :, :3], (R.T @ t)[None, :] + r[:, :, 3])
    return A, b


def residuals(M, mode, p_ref, p_cur, f, cam, rig):
    """float64 score of every correspondence under pose M (the oracle's formula)."""
    from oracle import ransac
    if mode == "euclid":
        return ransac.score_euclid(M, p_ref, p_cur)
    return ransac.score_bearing(M, p_ref, f, cam if rig is not None else None, rig)
