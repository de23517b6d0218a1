"""GPU parity: Arun solver, RANSAC (shared seeded hypothesis list) and refit vs the float64 oracle.
Inlier sets must be bit-exact; the data generator asserts a margin between every residual of the winning hypothesis
and the threshold (SURVEY §7 'hard parts' option b), and a clear winner, so float32 scoring cannot flip a decision."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import ransac

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, params=["tensor", "fma"])
def score_engine(request, monkeypatch):
    """Every test of this file runs with both engines of the scores, bearing and Euclidean: the bfloat16-split GEMMs on the
    tensor cores (csrc/score_mma.cuh, default) and the FP32-pipe kernel (SOS_SCORE_ENGINE=fma; the library reads the switch
    per call)."""
    if request.param == "fma":
        monkeypatch.setenv("SOS_SCORE_ENGINE", "fma")
    else:
        monkeypatch.delenv("SOS_SCORE_ENGINE", raising=False)
    return request.param


def dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def random_rotation(rng, max_deg):
    ax = rng.normal(size=3)
    ax /= np.linalg.norm(ax)
    a = np.deg2rad(rng.uniform(-max_deg, max_deg))
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    return np.eye(3) + np.sin(a) * K + (1 - np.cos(a)) * K @ K


def make_problem(rng, n, inlier_frac=0.35, sigma=0.005, rig=None):
    """3D-3D correspondences with a known motion: p_ref = R p_cur + t (+ noise); outliers are re-drawn points."""
    R = random_rotation(rng, 3.0)
    t = rng.normal(size=3) * 0.03
    p_cur = rng.normal(size=(n, 3))
    p_cur /= np.linalg.norm(p_cur, axis=1, keepdims=True)
    p_cur *= rng.uniform(0.5, 7.0, (n, 1))
    p_ref = p_cur @ R.T + t + rng.normal(0, sigma, (n, 3))
    out = rng.random(n) > inlier_frac
    p_ref[out] = rng.normal(size=(out.sum(), 3)) * 3
    cam = (rng.random(n) < 0.5).astype(np.uint8)
    cam.sort()
    if rig is None:
        f = p_cur / np.linalg.norm(p_cur, axis=1, keepdims=True)
    else:
        r = np.asarray(rig).reshape(-1, 3, 4)
        x = np.einsum("nji,nj->ni", r[cam, :, :3], p_cur - r[cam, :, 3])
        f = x / np.linalg.norm(x, axis=1, keepdims=True)
    f32 = lambda a: a.astype(np.float32)
    return f32(p_ref), f32(p_cur), f32(f), cam


def hyp_list(rng, H):
    return rng.integers(0, 2 ** 32, (H, 3), dtype=np.uint64).astype(np.uint32)


def as_i32(h):
    return dev(h.view(np.int32))


def test_arun_golden(ctx):
    g = load_golden("arun.npz")
    for k in (3, 4, 100):
        M, ok = ctx.arun_batch(dev(g[f"k{k}_v0"]), dev(g[f"k{k}_v1"]))
        assert ok.cpu().numpy().all()
        assert np.allclose(M.cpu().numpy(), g[f"k{k}_M"], rtol=0, atol=1e-9)
    # degenerate: collinear points
    v0 = np.zeros((2, 3, 3)); v0[:, 1, 0] = 1; v0[:, 2, 0] = 2
    M, ok = ctx.arun_batch(dev(v0), dev(v0.copy()))
    assert not ok.cpu().numpy().any()


@pytest.mark.parametrize("mode", ["euclid", "bearing", "bearing_rig"])
@pytest.mark.parametrize("n,H", [(300, 210), (2000, 512), (16000, 4096)])
def test_ransac_matches_oracle(ctx, mode, n, H):
    rng = np.random.default_rng(n + H + len(mode))
    rig = None
    if mode == "bearing_rig":
        Rc = random_rotation(rng, 10.0)
        rig = np.stack([np.hstack([np.eye(3), [[0.0], [0.0], [0.12]]]), np.hstack([Rc, [[0.01], [-0.02], [0.0]]])])
    B = 3
    thr = 0.05 if mode == "euclid" else 1.0 - np.cos(np.deg2rad(5.0))
    omode = "euclid" if mode == "euclid" else "bearing"
    probs = [make_problem(rng, n - 17 * b, rig=rig) for b in range(B)]
    cap = n
    p_ref = np.zeros((B, cap, 3), np.float32); p_cur = np.zeros_like(p_ref); f_cur = np.zeros_like(p_ref)
    cam = np.zeros((B, cap), np.uint8)
    ns = np.zeros(B, np.int32)
    for b, (a, c, f, cm) in enumerate(probs):
        ns[b] = len(a)
        p_ref[b, :len(a)], p_cur[b, :len(a)], f_cur[b, :len(a)], cam[b, :len(a)] = a, c, f, cm
    hyp = hyp_list(rng, H)
    hyp[3] = [5, 5, 7]             # repeated sample -> rejected
    hyp[4, 1] = hyp[4, 0]
    all_counts = torch.empty((B, H), dtype=torch.int32, device="cuda")
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(
        dev(p_ref), dev(p_cur), dev(ns), as_i32(hyp), 0 if mode == "euclid" else 1, thr,
        f_cur=dev(f_cur), cam=dev(cam) if rig is not None else None, rig=rig, n_cams=2 if rig is not None else 0,
        all_counts=all_counts)
    pose, best_hyp, best_count, mask, key = (x.cpu().numpy() for x in (pose, best_hyp, best_count, mask, key))
    all_counts = all_counts.cpu().numpy()
    for b, (a, c, f, cm) in enumerate(probs):
        o = ransac.ransac_p3d(a, c, hyp, omode, thr, f_cur=f, cam=cm if rig is not None else None, rig=rig)
        # the generator must give a decidable problem: clear winner and no residual on the threshold
        srt = np.sort(o["counts"])
        # the kernel re-decides every pair inside its float32 guard band in float64, so only residuals within
        # float64 rounding of the threshold could differ from the oracle
        assert o["margin"] > 1e-9, o["margin"]
        # EVERY hypothesis' inlier count equals the float64 oracle's, not only the winner's
        assert np.array_equal(np.where(all_counts[b] < 0, -1, all_counts[b]), o["counts"])
        assert best_hyp[b] == o["best_hyp"], (b, best_hyp[b], o["best_hyp"], srt[-3:])
        assert best_count[b] == o["best_count"]
        assert np.array_equal(mask[b, :ns[b]].astype(bool), o["mask"])
        assert not mask[b, ns[b]:].any()
        assert np.allclose(pose[b], o["pose"], rtol=1e-4, atol=1e-5)
        assert int(key[b]) >> 32 == o["best_count"] + 1
        assert o["counts"][3] == -1 and o["counts"][4] == -1
        assert o["best_count"] > 0.25 * ns[b]


def test_ransac_counts_all_hypotheses(ctx):
    """Every hypothesis' inlier count (not only the winner's) against the oracle, on margin-filtered data."""
    rng = np.random.default_rng(77)
    a, c, f, cm = make_problem(rng, 700)
    H = 256
    hyp = hyp_list(rng, H)
    o = ransac.ransac_p3d(a, c, hyp, "euclid", 0.05)
    # evaluate each hypothesis separately through the eval entry point
    B = H
    p_ref = np.broadcast_to(a, (B,) + a.shape).copy(); p_cur = np.broadcast_to(c, (B,) + c.shape).copy()
    ns = np.full(B, len(a), np.int32)
    pose, count, mask = ctx.ransac_p3d_eval(dev(p_ref), dev(p_cur), dev(ns), as_i32(hyp), 0, 0.05)
    count = count.cpu().numpy()
    got = np.where(count < 0, -1, count)
    rows = ransac.sample_rows(hyp, len(a))
    poses = ransac.arun_batch(c[rows].astype(np.float64), a[rows].astype(np.float64))
    near = 0
    for h in range(H):
        if o["counts"][h] < 0:
            assert got[h] == -1
            continue
        sc = ransac.score_euclid(poses[h], a.astype(np.float64), c.astype(np.float64))
        borderline = int(np.count_nonzero(np.abs(sc - 0.05) < 1e-5))
        near += borderline
        assert abs(int(got[h]) - int(o["counts"][h])) <= borderline
    assert near < H  # almost every hypothesis is decided exactly


def test_ransac_edge_cases(ctx):
    rng = np.random.default_rng(5)
    a, c, f, cm = make_problem(rng, 64)
    hyp = hyp_list(rng, 32)
    B, cap = 4, 64
    p_ref = np.zeros((B, cap, 3), np.float32); p_cur = np.zeros_like(p_ref)
    ns = np.array([64, 2, 0, 3], np.int32)
    p_ref[0], p_cur[0] = a, c
    p_ref[3, :3], p_cur[3, :3] = a[:3], c[:3]
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(dev(p_ref), dev(p_cur), dev(ns), as_i32(hyp), 0, 0.05)
    best_hyp, best_count, mask = best_hyp.cpu().numpy(), best_count.cpu().numpy(), mask.cpu().numpy()
    assert best_hyp[1] == -1 and best_count[1] == -1 and best_hyp[2] == -1 and not mask[1].any() and not mask[2].any()
    o0 = ransac.ransac_p3d(a, c, hyp, "euclid", 0.05)
    assert best_hyp[0] == o0["best_hyp"] and best_count[0] == o0["best_count"]
    o3 = ransac.ransac_p3d(a[:3], c[:3], hyp, "euclid", 0.05)
    assert best_hyp[3] == o3["best_hyp"] and best_count[3] == o3["best_count"]
    # zero hypotheses
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(dev(p_ref), dev(p_cur), dev(ns),
                                                          torch.zeros((0, 3), dtype=torch.int32, device="cuda"), 0, 0.05)
    assert (best_hyp.cpu().numpy() == -1).all()


def test_split_hypotheses_reduce_like_multi_gpu(ctx):
    """SURVEY §8e: splitting the hypothesis list and max-reducing the packed keys gives the single-list winner."""
    rng = np.random.default_rng(6)
    a, c, f, cm = make_problem(rng, 3000)
    H = 1024
    hyp = hyp_list(rng, H)
    args = (dev(a[None]), dev(c[None]), dev(np.array([len(a)], np.int32)))
    full = ctx.ransac_p3d(*args, as_i32(hyp), 0, 0.05)
    keys = []
    for r in range(4):
        part = ctx.ransac_p3d(*args, as_i32(hyp[r * 256:(r + 1) * 256]), 0, 0.05, hyp_offset=r * 256)
        keys.append(int(part[4].cpu().numpy()[0]))
    best = max(keys)
    assert best == int(full[4].cpu().numpy()[0])
    win = 0xFFFFFFFF - (best & 0xFFFFFFFF)
    assert win == int(full[1].cpu().numpy()[0])
    pose, count, mask = ctx.ransac_p3d_eval(*args, as_i32(hyp[win:win + 1]), 0, 0.05)
    assert int(count.cpu().numpy()[0]) == int(full[2].cpu().numpy()[0])
    assert np.array_equal(mask.cpu().numpy(), full[3].cpu().numpy())
    assert np.array_equal(pose.cpu().numpy(), full[0].cpu().numpy())


def test_refit_inliers(ctx):
    rng = np.random.default_rng(9)
    a, c, f, cm = make_problem(rng, 1500)
    hyp = hyp_list(rng, 300)
    args = (dev(a[None]), dev(c[None]), dev(np.array([len(a)], np.int32)))
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(*args, as_i32(hyp), 0, 0.05)
    refit, used = ctx.refit_inliers(args[0], args[1], mask, args[2])
    o = ransac.refit(a, c, mask.cpu().numpy()[0].astype(bool))
    assert int(used.cpu().numpy()[0]) == int(best_count.cpu().numpy()[0])
    assert np.allclose(refit.cpu().numpy()[0], o, rtol=1e-4, atol=1e-5)


def test_parallel_ransac_split_single_rank(ctx):
    """parallel.ransac_split with one rank must equal the plain call (the multi-rank path is exercised by
    scripts/bench_c4.py under torchrun and, for the reduce logic, by tests/test_parallel_cpu.py on gloo)."""
    from vo_single_camera_sos_b200 import parallel
    rng = np.random.default_rng(12)
    a, c, f, cm = make_problem(rng, 2500)
    hyp = hyp_list(rng, 700)
    args = (dev(a[None]), dev(c[None]), dev(np.array([len(a)], np.int32)))
    full = ctx.ransac_p3d(*args, as_i32(hyp), 0, 0.05)
    pose, count, mask, winner = parallel.ransac_split(ctx, *args, as_i32(hyp), 0, 0.05, rank=0, world=1)
    assert int(winner[0]) == int(full[1][0]) and int(count[0]) == int(full[2][0])
    assert torch.equal(mask, full[3]) and torch.equal(pose, full[0])
    # emulate 3 ranks on one GPU: keys of the slices, max, eval — what the NCCL all-reduce computes
    keys = []
    for r in range(3):
        lo, hi = parallel.shard_hypotheses(len(hyp), 3, r)
        keys.append(int(ctx.ransac_p3d(*args, as_i32(hyp[lo:hi]), 0, 0.05, hyp_offset=lo, want_mask=False)[4][0]))
    assert parallel.unpack_key(max(keys)) == (int(full[2][0]), int(full[1][0]))


@pytest.mark.parametrize("mode", ["euclid", "bearing"])
def test_long_hypothesis_list(ctx, mode):
    """More than 8192 hypotheses: the wide argmax block and several hypothesis tiles per problem; ties go to the lowest index."""
    rng = np.random.default_rng(5 + len(mode))
    n, H = 400, 9000
    a, c, f, cm = make_problem(rng, n)
    hyp = hyp_list(rng, H)
    hyp[8500] = hyp[17]            # the same triple twice: equal counts, the lower index must win if it is the best
    thr = 0.05 if mode == "euclid" else 1.0 - np.cos(np.deg2rad(5.0))
    all_counts = torch.empty((1, H), dtype=torch.int32, device="cuda")
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(dev(a[None]), dev(c[None]), dev(np.array([n], np.int32)), as_i32(hyp),
                                                           0 if mode == "euclid" else 1, thr, f_cur=dev(f[None]), all_counts=all_counts)
    o = ransac.ransac_p3d(a, c, hyp, mode, thr, f_cur=f)
    got = all_counts.cpu().numpy()[0]
    assert np.array_equal(np.where(got < 0, -1, got), o["counts"])
    assert int(best_hyp[0]) == o["best_hyp"] and int(best_count[0]) == o["best_count"]
    assert np.array_equal(mask.cpu().numpy()[0].astype(bool), o["mask"])
    assert int(key[0]) == ((o["best_count"] + 1) << 32) | (0xFFFFFFFF - o["best_hyp"])
