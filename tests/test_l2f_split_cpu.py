"""CPU: the float64 reference of the general float-descriptor L2 matcher (sos_l2f_top2) and the band of its tensor-core
ranking (oracle/l2f.py models csrc/hamming_mma.cu)."""
from fractions import Fraction

import numpy as np
import pytest

from conftest import load_golden
from oracle import hamming, l2f


def test_reference_equals_the_exact_integer_oracle_on_the_goldens():
    g = load_golden("l2.npz")
    for qk, tk in (("q", "t"), ("q64", "t64")):
        a, b = l2f.l2f_knn2(g[qk], g[tk]), hamming.l2_knn2(g[qk], g[tk])
        for x, y in zip(a, b):
            assert np.array_equal(x, y) and x.dtype == y.dtype
    for name, method, k, qk, tk in (("sift1", "SIFT", 1, "q", "t"), ("sift2", "SIFT", 2, "q", "t"), ("surf2", "SURF", 2, "q", "t"),
                                    ("surf1_64", "SURF", 1, "q64", "t64")):
        qi, ti, dd = l2f.l2f_match(g[qk], g[tk], method, k)
        assert np.array_equal(qi, g[f"{name}_q"]) and np.array_equal(ti, g[f"{name}_t"]) and np.array_equal(dd, g[f"{name}_d"])


def _exact_d2(q, t):
    return sum((Fraction(float(a)) - Fraction(float(b))) ** 2 for a, b in zip(q, t))


def test_reference_ranks_like_exact_arithmetic_where_float64_can_decide():
    rng = np.random.default_rng(5)
    for trial in range(40):
        dim = int(rng.choice([1, 3, 7, 16]))
        q = rng.normal(size=(1, dim)).astype(np.float32)
        t = np.repeat(q, 6, 0) + (rng.normal(size=(6, dim)) * 10.0 ** rng.integers(-7, 1)).astype(np.float32)
        t[3] = t[1]                                          # an exact tie
        t[4, 0] = np.nextafter(t[1, 0], np.float32(np.inf))   # one ulp away
        d64 = l2f.l2f_d2(q, t)[0]
        ex = [_exact_d2(q[0], r) for r in t]
        i0, _, i1, _ = l2f.l2f_knn2(q, t)
        for a in range(6):
            for b in range(6):
                # where the float64 values differ by more than their own rounding, the order is the exact order
                if abs(d64[a] - d64[b]) > 4 * (dim + 2) * 2.0 ** -53 * max(d64[a], d64[b]):
                    assert (d64[a] < d64[b]) == (ex[a] < ex[b])
        exact_order = sorted(range(6), key=lambda j: (ex[j], j))
        if all(abs(d64[j] - d64[k]) > 4 * (dim + 2) * 2.0 ** -53 * max(d64[j], d64[k]) or ex[j] == ex[k]
               for j in exact_order[:3] for k in exact_order[:3] if j != k):
            assert [i0[0], i1[0]] == exact_order[:2]


def _families(rng, dim):
    n = 64
    yield "gaussian", rng.normal(size=(n, dim)), rng.normal(size=(n, dim))
    a = rng.normal(size=(n, dim))
    yield "cancelling signs", a, -a + rng.normal(size=(n, dim)) * 1e-3
    d = rng.normal(size=(n, dim)) * 1e-4
    d[:, 0] = 1e3
    yield "one dominant component", d, rng.normal(size=(n, dim)) * 1e-4 + np.eye(1, dim) * 999.0
    # values whose mid piece is a float32 subnormal / bfloat16 flush: hi near 2^-120, mid below 2^-126
    yield "subnormal mid", (1 + rng.random((n, dim)) * 2 ** -7) * 2.0 ** -118, (1 + rng.random((n, dim))) * 2.0 ** -119
    # exactly halfway between two bfloat16 values (ties to even)
    h = (np.float32(1) + np.float32(2 ** -8) * (2 * rng.integers(0, 64, (n, dim)) + 1)) * np.sign(rng.normal(size=(n, dim)))
    yield "bfloat16 ties", h, h[::-1] * 0.75
    for mag in (1e-30, 1e-10, 1.0, 1e5, 1e15):
        yield f"magnitude {mag:g}", rng.normal(size=(n, dim)) * mag, rng.normal(size=(n, dim)) * mag * rng.random((n, 1))


@pytest.mark.parametrize("dim", [1, 7, 33, 64, 128])
@pytest.mark.parametrize("accum", ["rn16", "tz16"])
def test_key_model_stays_inside_the_band(dim, accum):
    rng = np.random.default_rng(dim)
    worst = 0.0
    for name, q, t in _families(rng, dim):
        q, t = q.astype(np.float32), t.astype(np.float32)
        a = l2f.l2f_key_model(q, t, accum).astype(np.float64)
        d2 = np.array([l2f.l2f_d2(q[i:i + 1], t[i:i + 1])[0, 0] for i in range(len(q))])
        qn2 = (q.astype(np.float64) ** 2).sum(1)
        m2 = (t.astype(np.float64) ** 2).sum(1).max()          # the segment's largest |t|^2
        band = l2f.l2f_band(qn2, m2)
        ratio = np.abs((qn2 - a) - d2) / band
        assert np.all(np.isfinite(a)), name
        assert ratio.max() <= 1.0, (name, ratio.max())
        worst = max(worst, ratio.max())
    assert worst <= 0.25, worst        # typical inputs sit far inside the worst case, as on the device


@pytest.mark.parametrize("accum", ["rn16", "tz16"])
def test_derived_worst_case_is_inside_the_band_constants(accum):
    for dim in (1, 16, 64, 65, 128):
        qt, tt, qq, lin, ab = l2f.worst_case_coefficients(dim, accum)
        assert qt < l2f.C_QT and tt < l2f.C_TT and qq < l2f.C_QQ and lin < l2f.C_LIN and ab < l2f.C_ABS, (dim, qt, tt, qq, lin, ab)
    qt, tt, *_ = l2f.worst_case_coefficients(128, "tz16")
    assert qt / l2f.C_QT > 0.95                       # the constant is the derivation, not a guess
