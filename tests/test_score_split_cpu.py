"""CPU: the arithmetic of the tensor-core score engine (bfloat16 three-way split, six partial products per feature, float32
accumulation) restated in NumPy — the split is exact, and the decision variable stays within a quarter of the engine's band."""
import numpy as np

from oracle import score_split as S
from oracle.ransac import arun_batch


def test_three_way_split_is_exact():
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.normal(size=20000) * 10.0 ** rng.integers(-6, 3, 20000), [0.0, 1.0, -1.0, 255.0, 1e-30, 3.0e38]]).astype(np.float32)
    h, m, l = S.split3(x)
    for piece in (h, m, l):
        assert np.array_equal(S.bf16_round(piece), piece)          # each piece is a bfloat16 value
    assert np.array_equal(((h.astype(np.float64) + m) + l).astype(np.float32), x)


def test_six_products_reproduce_the_float32_product():
    rng = np.random.default_rng(1)
    a = (rng.normal(size=(50000, 1)) * 7).astype(np.float32)
    b = (rng.normal(size=(50000, 1)) * 7).astype(np.float32)
    exact = a[:, 0].astype(np.float64) * b[:, 0].astype(np.float64)
    got = S.split_dot(a, b).astype(np.float64)
    # dropped ml, lm, ll (< 2^-25) and five float32 additions (2^-24 each): below 2^-21, like a short float32 FMA chain
    assert np.max(np.abs(got - exact) / np.abs(exact)) < 2.0 ** -21


def rot(rng, deg):
    ax = rng.normal(size=3); ax /= np.linalg.norm(ax)
    a = np.deg2rad(deg)
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def test_decision_variable_within_a_quarter_of_the_band():
    rng = np.random.default_rng(2)
    n = 400
    thr = 1.0 - np.cos(np.deg2rad(5.0))
    c2 = float(np.float32((1.0 - thr) ** 2))
    p = rng.normal(size=(n, 3)); p /= np.linalg.norm(p, axis=1, keepdims=True); p *= rng.uniform(0.5, 7.0, (n, 1))
    p = p.astype(np.float32)
    worst_b = worst_e = 0.0
    for trial in range(40):
        R = rot(rng, rng.uniform(0, 30)); t = rng.normal(size=3) * rng.choice([0.03, 0.5, 3.0])
        Rc = rot(rng, 10.0); tc = np.array([0.01, -0.02, 0.12])
        A = Rc.T @ R.T
        b = -Rc.T @ (R.T @ t + tc)
        x = p.astype(np.float64) @ A.T + b
        f = x / np.linalg.norm(x, axis=1, keepdims=True)
        f = (f + rng.normal(0, 0.05, f.shape)); f /= np.linalg.norm(f, axis=1, keepdims=True)
        f = f.astype(np.float32)
        bmax2 = float(b @ b)
        # bearing score: D = (s|s| + c^2 shift) - c^2 N'
        hs, hn = S.hypothesis_features(A, b, bmax2, bearing=True)
        cs, cn = S.correspondence_features(p, f, bearing=True)
        s = S.split_dot(hs[None, :], cs).astype(np.float64)
        N = S.split_dot(hn[None, :], cn).astype(np.float64) - S.B2_SHIFT * bmax2
        s_true = np.sum(f.astype(np.float64) * x, axis=1)
        n_true = np.sum(x * x, axis=1)
        scale = np.sum(p.astype(np.float64) ** 2, axis=1) + bmax2
        worst_b = max(worst_b, float(np.max(np.abs((s * np.abs(s) - c2 * N) - (s_true * np.abs(s_true) - c2 * n_true)) / scale)))
        # Euclidean score: r^2 = s' + n2 against the current-frame points q
        q = (x + rng.normal(0, 0.03, x.shape)).astype(np.float32)
        hs, hn = S.hypothesis_features(A, b, bmax2, bearing=False)
        cs, cn = S.correspondence_features(p, q, bearing=False)
        r2 = S.split_dot(hs[None, :], cs).astype(np.float64) + S.split_dot(hn[None, :], cn).astype(np.float64)
        r2_true = np.sum((x - q.astype(np.float64)) ** 2, axis=1)
        scale_e = scale + np.sum(q.astype(np.float64) ** 2, axis=1)
        worst_e = max(worst_e, float(np.max(np.abs(r2 - r2_true) / scale_e)))
    assert worst_b < S.BAND_REL / 4.0, worst_b
    assert worst_e < S.BAND_EUCLID / 4.0, worst_e


def model_errors(prob, mode, rig, accum, n_hyp=6):
    """Worst scaled error of the engine's (s, N') or r^2 under `accum` for a few poses from all-inlier-like triples of `prob`
    (the metric of tests/test_gpu_score_tc.py)."""
    import _score_families as F
    p_ref, p_cur, f, cam = (np.asarray(a) for a in prob)
    a64, c64, f64 = p_ref.astype(np.float64), p_cur.astype(np.float64), f.astype(np.float64)
    n = len(a64)
    rng = np.random.default_rng(n)
    rows = rng.choice(n, size=(n_hyp, 3), replace=False) if n_hyp * 3 <= n else rng.integers(0, n, (n_hyp, 3))
    poses = arun_batch(c64[rows], a64[rows])
    ci = cam.astype(np.int64) if rig is not None else np.zeros(n, np.int64)
    bearing = mode == "bearing"
    thr = F.THR_BEARING
    c2 = float(np.float32((1.0 - thr) ** 2))
    worst = 0.0
    for M in poses:
        A, b = F.pose_features(M, rig)
        b2 = np.sum(b * b, axis=1)
        bmax2 = float(np.max(b2))
        got_s, got_n = np.zeros(n), np.zeros(n)
        for c in range(len(A)):
            sel = ci == c
            if not sel.any():
                continue
            hs, hn = S.hypothesis_features(A[c], b[c], bmax2, bearing=bearing)
            cs, cn = S.correspondence_features(p_ref[sel], f[sel] if bearing else p_cur[sel], bearing=bearing)
            got_s[sel] = S.split_dot(hs[None, :], cs, accum).astype(np.float64)
            got_n[sel] = S.split_dot(hn[None, :], cn, accum).astype(np.float64)
        x = np.einsum("nik,nk->ni", A[ci], a64) + b[ci]
        if bearing:
            s, n2 = np.sum(f64 * x, axis=1), np.sum(x * x, axis=1)
            gn = got_n - S.B2_SHIFT * bmax2
            err = np.abs((got_s * np.abs(got_s) - c2 * gn) - (s * np.abs(s) - c2 * n2))
            scale = np.sum(a64 * a64, axis=1) + b2[ci]
        else:
            err = np.abs(got_s + got_n - np.sum((x - c64) ** 2, axis=1))
            scale = np.sum(a64 * a64, axis=1) + np.sum(c64 * c64, axis=1) + b2[ci]
        worst = max(worst, float(np.max(err / scale)))
    return worst


def test_families_within_a_quarter_of_the_band_per_instruction_rounding():
    """The adversarial families of tests/test_gpu_score_stress.py (and their millimetre versions) under the hardware model
    of the band's derivation — one rounding per MMA instruction of 16 products plus the accumulator, to nearest or toward
    zero: the decision variables stay within a quarter of the bands."""
    import _score_families as F
    rng = np.random.default_rng(5)
    report = []
    for family in F.FAMILIES:
        for mode in ("bearing", "bearing_rig", "euclid"):
            rig = F.rig_pair(rng) if mode == "bearing_rig" else None
            omode = "euclid" if mode == "euclid" else "bearing"
            prob = F.make(rng, family, 600, omode, rig=rig, exact_scale=True)
            band = S.BAND_EUCLID if omode == "euclid" else S.BAND_REL
            for scale in (1.0, 1000.0):
                p = F.scaled(prob, scale)
                for accum in ("rn16", "tz16"):
                    w = model_errors(p, omode, F.scaled_rig(rig, scale), accum)
                    report.append((family, mode, scale, accum, w / band))
    for r in report:
        print("%-14s %-12s x%-6g %s  %.3f of the band" % r)
    assert max(r[4] for r in report) < 0.25, max(report, key=lambda r: r[4])


def test_derived_worst_case_within_the_band():
    """The worst-case error model written in csrc/score_mma.cuh (feature rounding 2u, dropped split products 2u, and one
    rounding per MMA instruction, e = u to nearest or 2u toward zero; 5 instructions for s, 4 for n2) evaluated with its
    bounds on the sums of |terms|: it must stay inside the bands the kernel uses."""
    u = 2.0 ** -24
    for e in (u, 2 * u):
        ks, kn = 4 * u + 5 * e, 4 * u + 4 * e              # relative error of s (or s') and of n2 per unit of sum |terms|
        bearing = 6.2 * ks + 3.52 * kn + 22.8 * u            # x (|p|^2 + max |b|^2)
        euclid = 3.73 * ks + 2.0 * kn                        # x (|p|^2 + |q|^2 + |b|^2)
        assert bearing < S.BAND_REL and euclid < S.BAND_EUCLID, (e / u, bearing / S.BAND_REL, euclid / S.BAND_EUCLID)
