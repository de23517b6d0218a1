"""GPU: both engines of the RANSAC scores (csrc/score_mma.cuh and csrc/ransac.cu::score_kernel) against float64 at adversarial
geometry (tests/_score_families.py), in millimetres as well as metres, on the overflow branches of their deferred float64
paths, and at the benchmark's own sizes.

Every case checks all hypotheses' counts, the winner, its count and its inlier mask against oracle.ransac.ransac_p3d; on the
tensor-core engine it also bounds what the tensor cores accumulated against float64 through sos_ransac_score_probe, with the
metric of tests/test_gpu_score_tc.py, by a quarter of the engine's band.  The problems are built so that float64 decides every
pair: no residual of any hypothesis lies within 1e-12 relative of the threshold."""
import functools
import time

import numpy as np
import pytest
import torch

import _score_families as F
from oracle import ransac
from test_gpu_ransac import as_i32, dev, hyp_list, score_engine  # noqa: F401  (score_engine: both engines, autouse)
from test_gpu_score_tc import BAND_EUCLID, BAND_REL, B2_SHIFT, pack

pytestmark = pytest.mark.gpu

MODES = ["bearing", "bearing_rig", "euclid"]
# SOS_STAT_* of include/sosfront.h
TC_ITEMS, TC_CHUNKS, TC_CHUNKS_MAX, TC_IN_THREAD, TC_PAIRS, TC_ROUNDS_MAX, FMA_ENTRIES, FMA_OVERFLOW = range(8)
ECAP, PCAP, RS_QCAP = 1536, 2048, 2048    # csrc/score_mma.cuh, csrc/ransac.cu


def good_poses(prob, hyp, counts):
    p_ref, p_cur = prob[0].astype(np.float64), prob[1].astype(np.float64)
    rows = ransac.sample_rows(hyp, len(p_ref))
    good = np.nonzero(counts >= 0)[0]
    return good, ransac.arun_batch(p_cur[rows[good]], p_ref[rows[good]])


def assert_decidable(prob, hyp, counts, omode, thr, rig, chunk=512):
    """No float64 residual of any accepted hypothesis within 1e-12 relative of the threshold."""
    p_ref, p_cur, f = (a.astype(np.float64) for a in prob[:3])
    good, poses = good_poses(prob, hyp, counts)
    worst = np.inf
    for s in range(0, len(good), chunk):
        for M in poses[s:s + chunk]:
            r = F.residuals(M, omode, p_ref, p_cur, f, prob[3], rig)
            worst = min(worst, float(np.nanmin(np.abs(r - thr))) / thr)
    assert worst > 1e-12, worst


def run_and_check(ctx, probs, hyp, mode, thr, rig):
    """ransac_p3d on the current engine against the oracle; returns the oracle results."""
    omode = "euclid" if mode == "euclid" else "bearing"
    cams = rig is not None
    cap = max(len(p[0]) for p in probs)
    p_ref, p_cur, f_cur, cam, ns = pack(probs, cap)
    B, H = len(probs), len(hyp)
    all_counts = torch.empty((B, H), dtype=torch.int32, device="cuda")
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(
        dev(p_ref), dev(p_cur), dev(ns), as_i32(hyp), 0 if mode == "euclid" else 1, thr, f_cur=dev(f_cur),
        cam=dev(cam) if cams else None, rig=rig, n_cams=2 if cams else 0, all_counts=all_counts)
    all_counts, best_hyp, best_count, mask = (x.cpu().numpy() for x in (all_counts, best_hyp, best_count, mask))
    outs = []
    for b, (a, c, f, cm) in enumerate(probs):
        o = ransac.ransac_p3d(a, c, hyp, omode, thr, f_cur=f, cam=cm if cams else None, rig=rig)
        assert_decidable((a, c, f, cm), hyp, o["counts"], omode, thr, rig)
        assert np.array_equal(np.where(all_counts[b] < 0, -1, all_counts[b]), o["counts"]), b
        assert int(best_hyp[b]) == o["best_hyp"] and int(best_count[b]) == o["best_count"], b
        assert np.array_equal(mask[b, :len(a)].astype(bool), o["mask"]), b
        outs.append(o)
    return outs


def accumulator_error(ctx, probs, hyp, mode, thr, rig, outs):
    """Worst |err D| / (|p|^2 + |b|^2) (bearing) or |err r^2| / (|p|^2 + |q|^2 + |b|^2) (Euclidean) of the tensor cores'
    accumulators over every pair of every accepted hypothesis (the metric of tests/test_gpu_score_tc.py)."""
    cams = rig is not None
    cap = max(len(p[0]) for p in probs)
    p_ref, p_cur, f_cur, cam, ns = pack(probs, cap)
    counts, sn = ctx.ransac_score_probe(dev(p_ref), dev(p_cur), dev(f_cur) if mode != "euclid" else None, dev(ns), as_i32(hyp),
                                        thr, cam=dev(cam) if cams else None, rig=rig, n_cams=2 if cams else 0,
                                        score_mode=0 if mode == "euclid" else 1)
    counts, sn = counts.cpu().numpy(), sn.cpu().numpy().astype(np.float64)
    c2 = float(np.float32((1.0 - thr) ** 2))
    worst = 0.0
    for b, ((a, c, f, cm), o) in enumerate(zip(probs, outs)):
        assert np.array_equal(np.where(counts[b] < 0, -1, counts[b]), o["counts"]), b
        a64, c64, f64 = a.astype(np.float64), c.astype(np.float64), f.astype(np.float64)
        ci = cm.astype(np.int64) if cams else np.zeros(len(a), np.int64)
        good, poses = good_poses((a, c, f, cm), hyp, o["counts"])
        for h, M in zip(good, poses):
            A, bv = F.pose_features(M, rig)
            x = np.einsum("nik,nk->ni", A[ci], a64) + bv[ci]
            b2 = np.sum(bv * bv, axis=1)
            if mode == "euclid":
                truth = np.sum((x - c64) ** 2, axis=1)
                got = sn[b, h, :len(a), 0] + sn[b, h, :len(a), 1]
                scale = np.sum(a64 * a64, axis=1) + np.sum(c64 * c64, axis=1) + b2[ci]
            else:
                s, n2 = np.sum(f64 * x, axis=1), np.sum(x * x, axis=1)
                truth = s * np.abs(s) - c2 * n2
                gs, gn = sn[b, h, :len(a), 0], sn[b, h, :len(a), 1] - B2_SHIFT * float(np.max(b2))
                got = gs * np.abs(gs) - c2 * gn
                scale = np.sum(a64 * a64, axis=1) + b2[ci]
            worst = max(worst, float(np.max(np.abs(got - truth) / scale)))
    return worst


def family_case(rng, family, mode, n, B, exact_scale=False):
    rig = F.rig_pair(rng) if mode == "bearing_rig" else None
    omode = "euclid" if mode == "euclid" else "bearing"
    probs = [F.make(rng, family, n - 37 * b, omode, rig=rig, exact_scale=exact_scale) for b in range(B)]
    thr = F.THR_EUCLID if mode == "euclid" else F.THR_BEARING
    return probs, rig, thr


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", F.FAMILIES)
def test_families_match_float64(ctx, score_engine, family, mode):
    rng = np.random.default_rng([F.FAMILIES.index(family), MODES.index(mode)])
    probs, rig, thr = family_case(rng, family, mode, 1000, 2)
    hyp = hyp_list(rng, 384)
    outs = run_and_check(ctx, probs, hyp, mode, thr, rig)
    if score_engine == "tensor":
        band = BAND_EUCLID if mode == "euclid" else BAND_REL
        worst = accumulator_error(ctx, probs, hyp, mode, thr, rig, outs)
        print(f"\n{family}/{mode}: worst scaled accumulator error {worst:.3e} = {worst / band:.3f} of the band")
        assert worst < band / 4.0, (worst, band)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("family", F.FAMILIES)
def test_millimetres_count_like_metres(ctx, score_engine, family, mode):
    """The same problems with every length x 1000 (rig offsets 120 mm, Euclidean threshold 50 mm): the counts, the winner and
    the mask equal the float64 oracle's in both units, and the counts are the same."""
    rng = np.random.default_rng([7, F.FAMILIES.index(family), MODES.index(mode)])
    probs, rig, thr = family_case(rng, family, mode, 900, 2, exact_scale=True)
    hyp = hyp_list(rng, 256)
    outs_m = run_and_check(ctx, probs, hyp, mode, thr, rig)
    mm = [F.scaled(p, 1000.0) for p in probs]
    for p, q in zip(probs, mm):
        assert np.array_equal(p[0].astype(np.float64) * 1000.0, q[0].astype(np.float64))    # exactly the same problem
        assert np.array_equal(p[1].astype(np.float64) * 1000.0, q[1].astype(np.float64))
    thr_mm = thr * 1000.0 if mode == "euclid" else thr
    outs_mm = run_and_check(ctx, mm, hyp, mode, thr_mm, F.scaled_rig(rig, 1000.0))
    for o, p in zip(outs_m, outs_mm):
        assert np.array_equal(o["counts"], p["counts"]) and o["best_hyp"] == p["best_hyp"]
        assert np.array_equal(o["mask"], p["mask"])
    if score_engine == "tensor":
        band = BAND_EUCLID if mode == "euclid" else BAND_REL
        worst = accumulator_error(ctx, mm, hyp, mode, thr_mm, F.scaled_rig(rig, 1000.0), outs_mm)
        print(f"\n{family}/{mode} in mm: worst scaled accumulator error {worst:.3e} = {worst / band:.3f} of the band")
        assert worst < band / 4.0, (worst, band)


def far_field_batch(rng, B=4, n=1024):
    """Euclidean problems with |p| in 200 .. 1000 (thr 0.05): the tensor-core band, which grows with |p|^2, holds every pair
    of every good hypothesis, so each chunk of such a hypothesis is queued for the deferred pass.  97 % inliers (all others
    far off) keep 91 % of the hypotheses good, more than the 75 % of an item's chunk rows that fill its ECAP queue.  Two pairs
    per 32-correspondence batch are planted within 2 % of the threshold: the FP32 kernel's guard then holds a pair of nearly
    every (batch, good hypothesis), 7 000 of the 8 192 queue entries a block can produce, past its RS_QCAP of 2 048."""
    probs = []
    for b in range(B):
        R = F.rotation(rng, 20.0)
        t = rng.normal(size=3) * 0.3
        p_cur = F.unit(rng.normal(size=(n, 3))) * rng.uniform(200.0, 1000.0, (n, 1))
        p_ref = p_cur @ R.T + t
        out = rng.random(n) > 0.97
        p_ref[out] += rng.normal(size=(int(out.sum()), 3)) * 300.0
        plant = np.isin(np.arange(n) % 32, (7, 23)) & ~out
        k = int(plant.sum())
        p_ref[plant] += F.unit(rng.normal(size=(k, 3))) * F.THR_EUCLID * rng.uniform(0.98, 1.02, (k, 1))
        p_cur, p_ref = p_cur.astype(np.float32), p_ref.astype(np.float32)
        probs.append((p_ref, p_cur, np.zeros_like(p_cur), np.zeros(n, np.uint8)))
    return probs


def test_deferred_queues_overflow(ctx, score_engine):
    """The overflow branches of both deferred paths, shown to have run through the probe's counters: on the tensor-core
    engine more than ECAP queued chunks in an item (the rest decided in-thread) and several PCAP rounds; on the FP32 kernel
    blocks past RS_QCAP.  Counts, winners and masks equal float64.  B = 4, H = 9600, n = 1024 gives 75 hypothesis tiles x 2
    splits of the 8 correspondence tiles per problem on 148 SMs (launch_score_tc), 4 tiles = 2 048 chunk rows per item."""
    rng = np.random.default_rng(2024)
    probs = far_field_batch(rng)
    H = 9600
    hyp = hyp_list(rng, H)
    outs = run_and_check(ctx, probs, hyp, "euclid", F.THR_EUCLID, None)
    p_ref, p_cur, f_cur, cam, ns = pack(probs, 1024)
    stats = torch.zeros(8, dtype=torch.int32, device="cuda")
    args = (dev(p_ref), dev(p_cur), None, dev(ns), as_i32(hyp), F.THR_EUCLID)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    counts, _ = ctx.ransac_score_probe(*args, score_mode=0, want_sn=False, stats=stats)
    ev[1].record()
    torch.cuda.synchronize()
    st = stats.cpu().numpy()
    counts = counts.cpu().numpy()
    for b, o in enumerate(outs):
        assert np.array_equal(np.where(counts[b] < 0, -1, counts[b]), o["counts"]), b
    print(f"\n{score_engine}: stats {st.tolist()}, {ev[0].elapsed_time(ev[1]):.2f} ms for {len(probs)} x {H} x 1024 pairs")
    if score_engine == "tensor":
        assert st[TC_CHUNKS_MAX] > ECAP and st[TC_IN_THREAD] > 0
        assert st[TC_ROUNDS_MAX] >= 2 and st[TC_PAIRS] > PCAP
        assert st[FMA_ENTRIES] == 0
    else:
        assert st[FMA_OVERFLOW] > 0 and st[FMA_ENTRIES] > RS_QCAP
        assert st[TC_ITEMS] == 0


def test_probe_counters_on_an_ordinary_batch(ctx, score_engine):
    """On problems of the ordinary distribution nothing overflows, and the counters agree with themselves."""
    from test_gpu_ransac import make_problem
    rng = np.random.default_rng(11)
    probs = [make_problem(rng, 2000, inlier_frac=0.6, sigma=0.0) for _ in range(2)]
    p_ref, p_cur, f_cur, cam, ns = pack(probs, 2000)
    hyp = hyp_list(rng, 512)
    stats = torch.zeros(8, dtype=torch.int32, device="cuda")
    counts, sn = ctx.ransac_score_probe(dev(p_ref), dev(p_cur), dev(f_cur), dev(ns), as_i32(hyp), F.THR_BEARING,
                                        want_sn=False, stats=stats)
    st = stats.cpu().numpy()
    assert sn is None
    if score_engine == "tensor":
        assert st[TC_ITEMS] > 0 and st[TC_IN_THREAD] == 0 and st[TC_CHUNKS_MAX] <= ECAP
        assert (st[TC_PAIRS] > 0) == (st[TC_CHUNKS] > 0) and st[TC_PAIRS] <= 32 * st[TC_CHUNKS]
        assert st[FMA_ENTRIES] == 0 and st[FMA_OVERFLOW] == 0
    else:
        assert st[TC_ITEMS] == 0 and st[FMA_OVERFLOW] == 0
    counts = counts.cpu().numpy()
    for b, (a, c, f, cm) in enumerate(probs):
        o = ransac.ransac_p3d(a, c, hyp, "bearing", F.THR_BEARING, f_cur=f)
        assert np.array_equal(np.where(counts[b] < 0, -1, counts[b]), o["counts"])


def test_c2_moving_scene_stage_by_stage(ctx):
    """Config 2 at the benchmark's moving_fraction = 0.79 (about 35 % RANSAC inliers, the setting that sends pairs through the
    deferred path): every stage of two captured steps against the oracle."""
    from test_gpu_frontend import check_step, host
    from vo_single_camera_sos_b200 import ops, workload
    B = 2
    w = workload.build(ctx, "c2", batch=B, n_frames=2 * B, seed=5, score_mode=ops.SCORE_BEARING, moving_fraction=0.79)
    fe = w.frontend(ctx)
    prev = None
    for step in range(2):
        fr = workload.make_frames(w, step * B, B)
        fe.step(*workload.to_device(ctx, fr))
        torch.cuda.synchronize()
        buf = host(fe.buffers())
        prev = check_step(w, fr, buf, prev, "bearing")
    fe.close()


def c4_counts_float64(p_ref, p_cur, hyp, thr, hyp_idx=None, chunk=64):
    """Counts of the Euclidean score in float64 on the CPU (torch), for the hypotheses `hyp_idx` (all by default)."""
    n = len(p_ref)
    rows = ransac.sample_rows(hyp, n)
    H = len(hyp)
    idx = np.arange(H) if hyp_idx is None else np.asarray(hyp_idx)
    counts = np.full(len(idx), -1, np.int64)
    a64, c64 = p_ref.astype(np.float64), p_cur.astype(np.float64)
    r = rows[idx]
    ok = (r[:, 0] != r[:, 1]) & (r[:, 0] != r[:, 2]) & (r[:, 1] != r[:, 2])
    ok &= ~ransac.triangle_degenerate(c64[r]) & ~ransac.triangle_degenerate(a64[r])
    sel = np.nonzero(ok)[0]
    poses = ransac.arun_batch(c64[r[sel]], a64[r[sel]])
    A, C = torch.from_numpy(a64), torch.from_numpy(c64)
    closest = np.inf
    for s in range(0, len(sel), chunk):
        M = torch.from_numpy(poses[s:s + chunk])
        d = A[None] - (torch.einsum("hij,nj->hni", M[:, :, :3], C) + M[:, None, :, 3])
        res = torch.sqrt(torch.sum(d * d, dim=2))
        counts[sel[s:s + chunk]] = (res < thr).sum(dim=1).numpy()
        closest = min(closest, float(torch.min(torch.abs(res - thr))) / thr)
    return counts, closest


@functools.lru_cache(maxsize=1)
def c4_reference():
    """bench.c4_problem restated (50 000 correspondences x 65 536 hypotheses, 35 % inliers) and its float64 counts."""
    n, H = 50000, 65536
    rng = np.random.default_rng(4)
    p_cur = rng.normal(size=(1, n, 3))
    p_cur = (p_cur / np.linalg.norm(p_cur, axis=2, keepdims=True) * rng.uniform(0.5, 7.0, (1, n, 1))).astype(np.float32)
    ang = np.deg2rad(2.0)
    R = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]], np.float32)
    p_ref = (p_cur @ R.T + np.float32([0.03, -0.01, 0.02]) + rng.normal(0, 0.005, p_cur.shape)).astype(np.float32)
    out = rng.random(n) > 0.35
    p_ref[0, out] = (rng.normal(size=(int(out.sum()), 3)) * 3).astype(np.float32)
    hyp = rng.integers(0, 2 ** 32, (H, 3), dtype=np.uint64).astype(np.uint32)
    t0 = time.perf_counter()
    want, closest = c4_counts_float64(p_ref[0], p_cur[0], hyp, C4_THR)
    print(f"\nc4: float64 counts of {H} hypotheses on the CPU in {time.perf_counter() - t0:.1f} s; closest residual "
          f"{closest:.2e} relative of the threshold")
    return p_ref, p_cur, hyp, want, closest


C4_THR = 0.05


def test_c4_full_size_against_float64(ctx, score_engine):
    """Config 4 at full size (bench.py --workload c4: Euclidean score): every count, the winner and its mask against float64
    on the CPU, and parallel.ransac_split(world=1)."""
    from vo_single_camera_sos_b200 import ops, parallel
    p_ref, p_cur, hyp, want, closest = c4_reference()
    n, H, thr = p_ref.shape[1], len(hyp), C4_THR
    assert closest > 1e-12
    P_ref, P_cur, N = dev(p_ref), dev(p_cur), torch.tensor([n], dtype=torch.int32, device="cuda")
    all_counts = torch.empty((1, H), dtype=torch.int32, device="cuda")
    pose, best_hyp, best_count, mask, key = ctx.ransac_p3d(P_ref, P_cur, N, as_i32(hyp), ops.SCORE_EUCLID, thr, all_counts=all_counts)
    got = all_counts.cpu().numpy()[0]
    assert np.array_equal(np.where(got < 0, -1, got), want)
    o_best = int(np.argmax(want))
    assert int(best_hyp[0]) == o_best and int(best_count[0]) == int(want[o_best])
    rows = ransac.sample_rows(hyp[o_best:o_best + 1], n)
    M = ransac.arun_batch(p_cur[0][rows].astype(np.float64), p_ref[0][rows].astype(np.float64))[0]
    want_mask = ransac.score_euclid(M, p_ref[0].astype(np.float64), p_cur[0].astype(np.float64)) < thr
    assert np.array_equal(mask.cpu().numpy()[0].astype(bool), want_mask)
    spose, scount, smask, winner = parallel.ransac_split(ctx, P_ref, P_cur, N, as_i32(hyp), ops.SCORE_EUCLID, thr, rank=0, world=1)
    assert int(winner[0]) == o_best and int(scount[0]) == int(want[o_best])
    assert torch.equal(smask, mask) and torch.equal(spose, pose)
