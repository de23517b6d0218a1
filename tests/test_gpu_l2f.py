"""GPU: the general float-descriptor L2 matcher (sos_l2f_top2: split-bfloat16 tcgen05.mma ranking, float64 decision) against
its float64 reference (oracle/l2f.py) — indices and float32 distances bit for bit, with and without the second neighbour —
and against cv2.BFMatcher(NORM_L2) on live KAZE and RootSIFT descriptors within cv2's own float32 error."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import l2f

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run(ctx, qs, ts, want_second=True, stats=None):
    """All (q, t) pairs as the segments of one call -> per-segment (i0, d0, i1, d1) numpy arrays."""
    seg_q = np.concatenate([[0], np.cumsum([len(x) for x in qs])]).astype(np.int32)
    seg_t = np.concatenate([[0], np.cumsum([len(x) for x in ts])]).astype(np.int32)
    dim = (qs[0] if len(qs[0]) else ts[0]).shape[1]
    cat = lambda xs: np.concatenate([x.reshape(-1, dim) for x in xs]).astype(np.float32)
    out = ctx.l2f_top2(dev(cat(qs)), dev(cat(ts)), dev(seg_q[:-1]), dev(np.diff(seg_q)), dev(seg_t[:-1]), dev(np.diff(seg_t)),
                       max(1, int(np.diff(seg_q).max())), int(np.diff(seg_t).max()), want_second=want_second, stats=stats)
    out = [None if x is None else x.cpu().numpy() for x in out]
    return [tuple(None if x is None else x[seg_q[s]:seg_q[s + 1]] for x in out) for s in range(len(qs))]


def check(ctx, qs, ts, stats=None, what=""):
    for want_second in (True, False):
        res = run(ctx, qs, ts, want_second, stats)
        for s, (q, t) in enumerate(zip(qs, ts)):
            oi0, od0, oi1, od1 = l2f.l2f_knn2(q, t)
            i0, d0, i1, d1 = res[s]
            assert np.array_equal(i0, oi0), (what, s, want_second, np.nonzero(i0 != oi0)[0][:5])
            assert np.array_equal(d0.view(np.uint32), od0.view(np.uint32)), (what, s, want_second)
            if want_second:
                assert np.array_equal(i1, oi1), (what, s, np.nonzero(i1 != oi1)[0][:5])
                assert np.array_equal(d1.view(np.uint32), od1.view(np.uint32)), (what, s)
            else:
                assert i1 is None and d1 is None


def new_stats(ctx):
    from vo_single_camera_sos_b200 import ops
    return torch.zeros(ops.L2F_STATS, dtype=torch.int32, device="cuda")


def kinds(rng, n, dim):
    g = rng.normal(size=(n, dim))
    yield "gaussian", g.astype(np.float32)
    yield "unit (SURF-like)", (g / np.linalg.norm(g, axis=1, keepdims=True)).astype(np.float32)
    h = rng.gamma(0.7, 28.0, (n, dim))
    yield "RootSIFT-like", np.sqrt(h / h.sum(1, keepdims=True)).astype(np.float32)


def test_goldens_through_the_general_engine(ctx):
    g = load_golden("l2.npz")
    from oracle import hamming
    for qk, tk in (("q", "t"), ("q64", "t64")):
        for want_second in (True, False):
            i0, d0, i1, d1 = run(ctx, [g[qk]], [g[tk]], want_second)[0]
            oi0, od0, oi1, od1 = hamming.l2_knn2(g[qk], g[tk])             # cv2's own results on these inputs
            assert np.array_equal(i0, oi0) and np.array_equal(d0, od0)
            if want_second:
                assert np.array_equal(i1, oi1) and np.array_equal(d1, od1)


@pytest.mark.parametrize("dim", [128, 64, 33, 7, 1])
def test_ragged_segments_against_the_float64_reference(ctx, dim):
    rng = np.random.default_rng(dim)
    sizes = [(700, 900), (130, 513), (257, 128), (5, 1300), (0, 10), (40, 0), (1, 1)]
    for k in range(3):
        qs, ts, what = [], [], None
        for nq, nt in sizes:
            what, base = list(kinds(rng, nq + nt, dim))[k]
            q = (base[:nq] + 0.05 * rng.normal(size=(nq, dim))).astype(np.float32) if k == 0 else base[:nq]
            t = base[nq:].copy()
            if nq and nt > 300:                     # winners duplicated into a later tile and into the last split
                i0 = l2f.l2f_knn2(q[:30], t)[0]
                for j in range(0, len(i0), 3):
                    if i0[j] + 130 < nt:
                        t[i0[j] + 130] = t[i0[j]]
                t[nt - 1] = t[i0[-1]]
            qs.append(q); ts.append(t)
        check(ctx, qs, ts, what=(dim, what))


def _frames():
    import cv2
    rng = np.random.default_rng(21)
    img = cv2.GaussianBlur((rng.random((480, 640)) * 255).astype(np.uint8), (0, 0), 2.0)
    img = cv2.normalize(img, None, 0, 255, cv2.NORM_MINMAX)
    for _ in range(60):
        c = tuple(int(x) for x in rng.integers(0, [640, 480]))
        cv2.circle(img, c, int(rng.integers(4, 30)), int(rng.integers(0, 255)), -1)
    rot = cv2.warpAffine(img, cv2.getRotationMatrix2D((320, 240), 12.0, 1.05), (640, 480))
    return img, rot


def test_real_descriptors_against_the_reference_and_cv2(ctx):
    import cv2
    a, b = _frames()
    sets = []
    kaze = cv2.KAZE_create()
    sets.append(("KAZE", kaze.detectAndCompute(a, None)[1], kaze.detectAndCompute(b, None)[1]))
    sift = cv2.SIFT_create(nfeatures=1500)
    root = lambda d: np.sqrt(d / np.maximum(d.sum(1, keepdims=True), 1e-12)).astype(np.float32)
    sets.append(("RootSIFT", root(sift.detectAndCompute(a, None)[1]), root(sift.detectAndCompute(b, None)[1])))
    stats = new_stats(ctx)
    for name, q, t in sets:
        assert len(q) > 200 and len(t) > 200 and not np.array_equal(q, np.round(q)), name
        check(ctx, [q], [t], stats=stats, what=name)
        i0, d0, i1, d1 = run(ctx, [q], [t])[0]
        m = cv2.BFMatcher(cv2.NORM_L2).knnMatch(q, t, k=2)
        ci = np.array([[x.trainIdx for x in p] for p in m])
        cd = np.array([[x.distance for x in p] for p in m], np.float64)
        d2 = l2f.l2f_d2(q, t)
        d2.sort(axis=1)
        # cv2 sums float32 squares in a build-dependent order: |error of d^2| <= dim 2^-24 d^2 (+ one rounding of sqrt)
        gam = q.shape[1] * 2.0 ** -24
        sure = (d2[:, 1] - d2[:, 0] > 2.1 * gam * d2[:, 1]) & (d2[:, 2] - d2[:, 1] > 2.1 * gam * d2[:, 2])
        assert sure.mean() > 0.9, name
        assert np.array_equal(ci[sure, 0], i0[sure]) and np.array_equal(ci[sure, 1], i1[sure]), name
        for c, d in ((cd[:, 0], d0), (cd[:, 1], d1)):
            assert np.all(np.abs(c - d) <= (gam + 2.0 ** -23) * d + 1e-30), name


def test_queries_the_band_cannot_decide_are_redecided_in_float64(ctx):
    rng = np.random.default_rng(8)
    # every train row equal: every query is a tie, neighbours 0 and 1
    q = rng.normal(size=(300, 64)).astype(np.float32)
    t = np.repeat(rng.normal(size=(1, 64)).astype(np.float32), 700, 0)
    stats = new_stats(ctx)
    i0, d0, i1, d1 = run(ctx, [q], [t], True, stats)[0]
    assert (i0 == 0).all() and (i1 == 1).all()
    assert int(stats[0]) == len(q)
    check(ctx, [q], [t])
    # near-duplicates one ulp apart in one component
    t = np.repeat(q[:50], 6, 0)
    for j in range(0, len(t), 6):
        t[j + 1, 7] = np.nextafter(t[j + 1, 7], np.float32(np.inf))
        t[j + 3, 0] = np.nextafter(t[j + 3, 0], np.float32(-np.inf))
    t = t[rng.permutation(len(t))]
    check(ctx, [q], [t], what="one ulp")
    # magnitudes whose float32 products underflow / overflow in the accumulators
    for mag in (1e-30, 1e20, 1e37):
        qm = (rng.normal(size=(200, 128)) * mag).astype(np.float32)
        tm = np.concatenate([(rng.normal(size=(300, 128)) * mag).astype(np.float32), qm[:20] * np.float32(0.999)])
        assert np.all(np.isfinite(qm)) and np.all(np.isfinite(tm))
        stats = new_stats(ctx)
        check(ctx, [qm], [tm], stats=stats, what=mag)
        assert int(stats[0]) > 0
    # zero vectors and -0.0
    z = np.zeros((20, 33), np.float32)
    z[10:] = -0.0
    tz = np.concatenate([np.full((5, 33), -0.0, np.float32), rng.normal(size=(200, 33)).astype(np.float32), np.zeros((5, 33), np.float32)])
    check(ctx, [z, rng.normal(size=(40, 33)).astype(np.float32)], [tz, tz], what="zeros")


def test_non_finite_values_are_refused(ctx):
    q = np.ones((300, 64), np.float32)
    t = np.zeros((400, 64), np.float32)
    for bad in (np.nan, np.inf, -np.inf):
        for side in (0, 1):
            a, b = q.copy(), t.copy()
            (a, b)[side][5, 7] = bad
            with pytest.raises(ValueError):
                run(ctx, [a], [b])


def test_full_size_against_the_float64_reference(ctx):
    rng = np.random.default_rng(77)
    h = rng.gamma(0.7, 28.0, (8000 + 8000 + 24 * 700, 128))
    x = np.sqrt(h / h.sum(1, keepdims=True)).astype(np.float32)
    big_t = x[:8000]
    big_q = (big_t[rng.permutation(8000)] + 0.02 * rng.normal(size=(8000, 128))).astype(np.float32)
    qs, ts = [big_q], [big_t]
    for s in range(12):
        b = x[16000 + s * 1400:16000 + (s + 1) * 1400]
        n = 650 + 10 * s
        qs.append((b[:n] + 0.02 * rng.normal(size=(n, 128))).astype(np.float32)); ts.append(b[700:700 + n])
    stats = new_stats(ctx)
    res = run(ctx, qs, ts, True, stats)
    for s, (q, t) in enumerate(zip(qs, ts)):
        oi0, od0, oi1, od1 = l2f.l2f_knn2(q, t, block=512)
        i0, d0, i1, d1 = res[s]
        assert np.array_equal(i0, oi0) and np.array_equal(i1, oi1), s
        assert np.array_equal(d0, od0) and np.array_equal(d1, od1), s
    assert int(stats[1]) <= 250000, int(stats[1])           # the error stays below a quarter of the band
    assert int(stats[0]) < 0.2 * sum(len(q) for q in qs)


def test_mirror_picks_the_engine_from_the_values(ctx):
    from omnistereo.camera_models import FeatureMatcher
    from vo_single_camera_sos_b200.omnistereo import device_context
    rng = np.random.default_rng(4)
    for dim in (64, 128):
        h = rng.gamma(0.7, 28.0, (900, dim))
        x = np.sqrt(h / h.sum(1, keepdims=True)).astype(np.float32)
        q, t = (x[:400] + 0.01 * rng.normal(size=(400, dim))).astype(np.float32), x[400:]
        for method, k in (("SURF", 1), ("SURF", 2), ("SIFT", 2)):
            qi, ti, dd = FeatureMatcher(method, "BF", k).match_arrays(q, t)
            oq, ot, od = l2f.l2f_match(q, t, method, k)
            assert np.array_equal(qi, oq) and np.array_equal(ti, ot) and np.array_equal(dd, od), (dim, method, k)
    g = load_golden("l2.npz")
    c = device_context()
    c.profile_begin()
    FeatureMatcher("SIFT", "BF", 2).match_arrays(g["q"], g["t"])
    names = [n.split("#")[0] for n, _ in c.profile_end()]
    assert "l2_mma_kernel" in names and not any(n.startswith("l2f_") for n in names), names
    c.profile_begin()
    FeatureMatcher("SIFT", "BF", 2).match_arrays(g["q"] + np.float32(0.5), g["t"])
    names = [n.split("#")[0] for n, _ in c.profile_end()]
    assert "l2f_mma_kernel" in names and "l2_mma_kernel" not in names, names
    with pytest.raises(ValueError):
        FeatureMatcher("SURF", "BF", 1).match_arrays(np.full((3, 64), np.nan, np.float32), t[:, :64])
