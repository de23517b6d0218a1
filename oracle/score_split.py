"""Oracle for the tensor-core score engine's arithmetic (csrc/score_mma.cuh). TEST INFRASTRUCTURE ONLY — see oracle/__init__.py.

The engine evaluates the reference's bearing score (pose_est_tools.py:150-203, non-central correction :181-185) as two small-K
GEMMs in bfloat16: every float32 feature is split into three bfloat16 pieces and six partial products per feature are
accumulated in float32.  This module restates that arithmetic in NumPy (bfloat16 rounding emulated on the bit pattern,
float32 accumulation in the order of the K columns, or one rounding per MMA instruction of 16 columns), so that the split's
exactness and the size of the guard band can be checked without a GPU.  The tensor core's internal accumulation is not
specified; the GPU tests (tests/test_gpu_score_tc.py, tests/test_gpu_score_stress.py) measure the real thing."""
from __future__ import annotations

import numpy as np

BAND_REL = 13.0 * 2.0 ** -20 + 5e-7      # csrc/score_mma.cuh
B2_SHIFT = 1.52
BAND_EUCLID = 5e-6


def bf16_round(x: np.ndarray) -> np.ndarray:
    """float32 -> nearest bfloat16 (ties to even), returned as float32."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return (r & 0xFFFFFFFF).astype(np.uint32).view(np.float32)


def split3(x: np.ndarray):
    """x == h + m + l exactly, each a bfloat16 value (score_mma.cuh::split3)."""
    x = np.asarray(x, np.float32)
    h = bf16_round(x)
    r1 = (x - h).astype(np.float32)
    m = bf16_round(r1)
    r2 = (r1 - m).astype(np.float32)
    l = bf16_round(r2)
    return h, m, l


def round_f32(x: np.ndarray, mode: str) -> np.ndarray:
    """float64 -> float32, to nearest ("rn") or toward zero ("tz")."""
    f = np.asarray(x, np.float64).astype(np.float32)
    if mode == "tz":
        over = np.abs(f.astype(np.float64)) > np.abs(x)
        f[over] = np.nextafter(f[over], np.float32(0))
    return f


def split_dot(a: np.ndarray, b: np.ndarray, accum: str = "column") -> np.ndarray:
    """sum_k a[..., k] * b[..., k] the way the engine forms it: per feature the six products hh, hm, mh, hl, lh, mm (each exact
    in float32: 8 x 8 mantissa bits), laid out as six consecutive K columns per feature.
    accum = "column": float32 accumulation column by column (one rounding per product);
    accum = "rn16" / "tz16": one rounding per MMA instruction, to nearest / toward zero — the accumulator plus the exact sum
    of the instruction's 16 K columns (the zero padding of the last one included), which is the hardware model of the band's
    derivation (csrc/score_mma.cuh)."""
    ah, am, al = split3(a)
    bh, bm, bl = split3(b)
    shape = np.broadcast_shapes(a.shape, b.shape)[:-1]
    if accum == "column":
        acc = np.zeros(shape, np.float32)
        for k in range(a.shape[-1]):
            for x, y in ((ah, bh), (ah, bm), (am, bh), (ah, bl), (al, bh), (am, bm)):
                acc = (acc + (x[..., k] * y[..., k]).astype(np.float32)).astype(np.float32)
        return acc
    if accum not in ("rn16", "tz16"):
        raise ValueError(accum)
    prods = [x[..., k].astype(np.float64) * y[..., k].astype(np.float64)
             for k in range(a.shape[-1]) for x, y in ((ah, bh), (ah, bm), (am, bh), (ah, bl), (al, bh), (am, bm))]
    acc = np.zeros(shape, np.float32)
    for s in range(0, len(prods), 16):
        tot = acc.astype(np.float64)
        for pr in prods[s:s + 16]:   # products of two bfloat16 values: the float64 sum of 17 terms is exact to 2^-50 or so
            tot = tot + pr
        acc = round_f32(tot, accum[:2])
    return acc


def hypothesis_features(A: np.ndarray, b: np.ndarray, bmax2: float, bearing: bool = True):
    """(fs[13], fn[10]) of one hypothesis and camera: A (3x3) and b (3) in float64 (emit_hyp_row)."""
    fs = np.concatenate([A.reshape(9), b, [1.0]]).astype(np.float32)
    G = A.T @ A
    v = A.T @ b
    fn = np.array([G[0, 0], G[1, 1], G[2, 2], G[0, 1], G[0, 2], G[1, 2], v[0], v[1], v[2],
                   b @ b + (B2_SHIFT * bmax2 if bearing else 0.0)]).astype(np.float32)
    return fs, fn


def correspondence_features(p: np.ndarray, f: np.ndarray, bearing: bool = True):
    """(fs[n,13], fn[n,10]) of correspondences: p = reference points, f = bearings (bearing score) or current points (Euclidean)."""
    p = np.asarray(p, np.float64)
    f = np.asarray(f, np.float64)
    sc = 1.0 if bearing else -2.0
    fs = np.concatenate([(sc * f[:, :, None] * p[:, None, :]).reshape(len(p), 9), sc * f,
                         np.zeros((len(p), 1)) if bearing else np.sum(f * f, axis=1, keepdims=True)], axis=1).astype(np.float32)
    fn = np.stack([p[:, 0] ** 2, p[:, 1] ** 2, p[:, 2] ** 2, 2 * p[:, 0] * p[:, 1], 2 * p[:, 0] * p[:, 2], 2 * p[:, 1] * p[:, 2],
                   2 * p[:, 0], 2 * p[:, 1], 2 * p[:, 2], np.ones(len(p))], axis=1).astype(np.float32)
    return fs, fn
