"""Oracle for the general float-descriptor L2 matcher (sos_l2f_top2, csrc/hamming_mma.cu). TEST INFRASTRUCTURE ONLY — see
oracle/__init__.py.

Two things live here:
  * the float64 reference that defines the matcher's results: d^2(q, t) = sum_k (double(q_k) - double(t_k))^2, summed for
    k = 0 .. dim-1 in order with separate roundings of the subtraction, the product and the sum (no FMA); the two smallest
    d^2 per query with ties to the lowest train row; distance = float32(sqrt(d^2)).  On integer-valued descriptors in
    [0, 255] this is cv2.BFMatcher(NORM_L2) exactly (oracle/hamming.py::l2_knn2);
  * a NumPy model of the engine's approximate key a ~ 2 <q, t> - |t|^2 (two-piece bfloat16 split, hi*hi + hi*mid + mid*hi,
    three bfloat16 pieces of |t|^2, one float32 rounding per MMA instruction) and of the band B_q that bounds
    |a - (|q|^2 - d^2)|, so that the band can be checked without a GPU."""
from __future__ import annotations

import numpy as np

from .score_split import bf16_round, round_f32

# csrc/hamming_mma.cu: B_q = C_QT |q| M + C_TT M^2 + C_QQ |q|^2 + C_LIN (|q| + M) + C_ABS, M = the segment's largest |t|
C_QT, C_TT, C_QQ = 1e-4, 4e-6, 1e-13
C_LIN, C_ABS = 2.0 ** -118, 2.0 ** -116
TINY = np.float32(2.0 ** -126)


# ---- the reference ----------------------------------------------------------------------------------------------------
def l2f_d2(q: np.ndarray, t: np.ndarray) -> np.ndarray:
    """[nq, nt] float64 squared distances in the contract's order (vectorised over rows, a loop over k)."""
    q = np.asarray(q, np.float32).astype(np.float64)
    t = np.asarray(t, np.float32).astype(np.float64)
    acc = np.zeros((q.shape[0], t.shape[0]))
    for k in range(q.shape[1]):
        d = q[:, k, None] - t[None, :, k]
        acc = acc + d * d
    return acc


def l2f_knn2(q: np.ndarray, t: np.ndarray, block: int = 1024):
    """Two nearest train rows per query by (d^2, train index) -> (idx0, d0, idx1, d1); missing neighbours are -1."""
    nq, nt = len(q), len(t)
    idx = np.full((nq, 2), -1, np.int32)
    dist = np.full((nq, 2), -1.0, np.float32)
    if nq == 0 or nt == 0:
        return idx[:, 0], dist[:, 0], idx[:, 1], dist[:, 1]
    for a in range(0, nq, block):
        d2 = l2f_d2(q[a:a + block], t)
        rows = np.arange(d2.shape[0])
        i0 = np.argmin(d2, axis=1)                     # first occurrence: ties to the lowest train row
        idx[a:a + block, 0] = i0
        dist[a:a + block, 0] = np.sqrt(d2[rows, i0]).astype(np.float32)
        if nt > 1:
            d2[rows, i0] = np.inf
            i1 = np.argmin(d2, axis=1)
            idx[a:a + block, 1] = i1
            dist[a:a + block, 1] = np.sqrt(d2[rows, i1]).astype(np.float32)
    return idx[:, 0], dist[:, 0], idx[:, 1], dist[:, 1]


def l2f_match(q, t, method="SURF", k_best=1):
    """FeatureMatcher(method, "BF", k_best).match on float descriptors with the reference above -> (query_idx, train_idx,
    distance float32) in the output order of oracle/hamming.py::l2_match."""
    i0, d0, i1, d1 = l2f_knn2(q, t)
    qi = np.arange(len(q), dtype=np.int32)
    if k_best == 2 and method.upper() == "SIFT":
        keep = (i1 >= 0) & (d0.astype(np.float64) < d1.astype(np.float64) * 0.75)
        qi, ti, dd = qi[keep], i0[keep], d0[keep]
    elif k_best == 2:
        qi = np.repeat(qi, 2)
        ti, dd = np.stack([i0, i1], 1).reshape(-1), np.stack([d0, d1], 1).reshape(-1)
        have = ti >= 0
        qi, ti, dd = qi[have], ti[have], dd[have]
    else:
        ti, dd = i0, d0
    order = np.argsort(dd, kind="stable")
    return qi[order], ti[order], dd[order]


# ---- the engine's arithmetic ------------------------------------------------------------------------------------------
def _flush(x: np.ndarray) -> np.ndarray:
    x = np.asarray(x, np.float32).copy()
    x[np.abs(x) < TINY] = 0
    return x


def split2(x: np.ndarray):
    """x ~ hi + mid: hi = bf16(x), mid = bf16(x - hi), pieces below 2^-126 set to 0 (l2f_bf16 in hamming_mma.cu)."""
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        hi = _flush(bf16_round(x))
        mid = _flush(bf16_round((x - hi).astype(np.float32)))
    return hi, mid


def norm_pieces(t: np.ndarray):
    """|t|^2 (float64) and its three bfloat16 pieces, as the expansion forms them."""
    n = (np.asarray(t, np.float64) ** 2).sum(-1)
    n1 = _flush(bf16_round(n.astype(np.float32)))
    r1 = n - n1.astype(np.float64)
    n2 = _flush(bf16_round(r1.astype(np.float32)))
    n3 = _flush(bf16_round((r1 - n2.astype(np.float64)).astype(np.float32)))
    return n, n1, n2, n3


def l2f_key_model(q: np.ndarray, t: np.ndarray, accum: str = "rn16") -> np.ndarray:
    """The engine's float32 accumulator for paired rows q[i], t[i] ([n, dim] each): one instruction for the |t|^2 pieces,
    then per 16-value block the instructions hi*hi, hi*mid, mid*hi (the device's issue order), each adding the exact sum of
    its 16 products to the accumulator and rounding once, to nearest ("rn16") or toward zero ("tz16")."""
    mode = {"rn16": "rn", "tz16": "tz"}[accum]
    q = np.asarray(q, np.float32)
    t = np.asarray(t, np.float32)
    qh, qm = split2(q)
    th, tm = split2(t)
    qh, qm = 2 * qh.astype(np.float64), 2 * qm.astype(np.float64)
    th, tm = th.astype(np.float64), tm.astype(np.float64)
    _, n1, n2, n3 = norm_pieces(t)
    acc = round_f32(-(n1.astype(np.float64) + n2 + n3), mode)
    dim = q.shape[1]
    for k0 in range(0, dim, 16):
        sl = slice(k0, min(dim, k0 + 16))
        for a, b in ((qh, th), (qh, tm), (qm, th)):
            acc = round_f32(acc.astype(np.float64) + (a[:, sl] * b[:, sl]).sum(1), mode)
    return acc


def l2f_band(qn2, m2):
    """B_q from |q|^2 and the segment's max |t|^2 (both float64), as l2f_decide_kernel computes it."""
    qn, mt = np.sqrt(qn2), np.sqrt(m2)
    return C_QT * qn * mt + C_TT * m2 + C_QQ * qn2 + C_LIN * (qn + mt) + C_ABS


def worst_case_coefficients(dim: int, accum: str):
    """The derivation's worst case (hamming_mma.cu) as coefficients of (|q| M, M^2, |q|^2, |q| + M, 1) for one dim."""
    u, e = 2.0 ** -24, (2.0 ** -24 if accum == "rn16" else 2.0 ** -23)
    b = 2.0 ** -8
    m = 3 * -(-dim // 16) + 1                                     # MMA instructions
    split = 2 * ((1 + b) * 2.0 ** -16 + (b * (1 + b)) ** 2 + 2.0 ** -16 * (1 + b) + 3 * 2.0 ** -24)
    t_qt = 2 * (1 + b) ** 2 * (1 + 2 * b * (1 + b))               # sum of |terms| per |q_k| |t_k|
    t_tt = (1 + b) * (1 + b * (1 + b)) * 1.0002
    ref = (dim + 3) * 2.0 ** -53
    qt = split + m * e * t_qt + 2 * ref
    tt = 1.0002 * u + m * e * t_tt + ref
    qq = 2 * ref
    lin = 2.01 * 2.0 ** -125 * np.sqrt(dim) * 2
    ab = (3 * dim + 3 + m) * 2.0 ** -126 + 3 * 2.0 ** -126
    return qt, tt, qq, lin, ab
