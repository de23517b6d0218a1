#!/usr/bin/env python
"""Kernel micro-benchmarks at C2 sizes (CUDA events, warm-up, inputs rotated): python scripts/kbench.py [hamming|ransac|remap|dense|rgbd|l2|all]

Prints one JSON line per kernel and input variant.
"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vo_single_camera_sos_b200 import ops  # noqa: E402


def timeit(fn, iters=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def bench_hamming(ctx, popc_peak, n=4500, segs=32, top2=False):
    g = torch.Generator(device="cuda").manual_seed(1)
    cap = 8192
    q = torch.randint(0, 256, (segs * cap, 32), dtype=torch.uint8, device="cuda", generator=g)
    t = torch.randint(0, 256, (segs * cap, 32), dtype=torch.uint8, device="cuda", generator=g)
    start = (torch.arange(segs, device="cuda", dtype=torch.int32) * cap).contiguous()
    ln = torch.full((segs,), n, dtype=torch.int32, device="cuda")
    out = ctx.hamming_top2(q, t, start, ln, start, ln, cap, cap, want_second=top2)
    ms = timeit(lambda: ctx.hamming_top2(q, t, start, ln, start, ln, cap, cap, want_second=top2, out=out))
    pairs = segs * n * n
    tp = pairs * 8 / (ms * 1e-3) / 1e12
    return dict(kernel="hamming", top2=top2, ms=ms,
                pairs_per_s=pairs / (ms * 1e-3), tpopc_equiv=tp, frac_of_popc_peak=tp / popc_peak)


def bench_dense(ctx, hbm_peak, B=16, rows=849, cols=2400):
    """Dense triangulation (SURVEY §8f N4): 4 B disparity in, 12 B xyz + 1 B valid out per panorama pixel."""
    from vo_single_camera_sos_b200 import synth
    rig = synth.make_rig(2048, 2048, cols, seed=0)
    rows = rig.pano["rows"]
    g = torch.Generator(device="cuda").manual_seed(5)
    disp = [torch.rand((B, rows, cols), device="cuda", generator=g) * 40.0 for _ in range(2)]
    for d in disp:
        d[d < 6.0] = 0.0
    out = ctx.dense_triangulate(rig.pano_vector(), rig.pano_vector(), disp[0], rig.f_top, rig.f_bot, 1.0, 64.0, rows - 1.0)
    it = [0]

    def run():
        ctx.dense_triangulate(rig.pano_vector(), rig.pano_vector(), disp[it[0] & 1], rig.f_top, rig.f_bot, 1.0, 64.0, rows - 1.0,
                              out=out)
        it[0] += 1
    ms_call = timeit(run)          # per call incl. host overhead of the wrapper
    ctx.profile_begin()            # per launch, CUDA events on the launching stream
    for _ in range(20):
        run()
    marks = ctx.profile_end()
    per = {"column_table": [t for _, t in marks[0::2]], "dense": [t for _, t in marks[1::2]]}   # two launches per call
    ms = float(np.median(per["dense"]))
    nbytes = B * rows * cols * 17
    return dict(kernel="dense_triangulate", ms=ms, ms_per_call=ms_call, pixels=B * rows * cols, gbps=nbytes / (ms * 1e-3) / 1e9,
                frac_of_hbm_peak=nbytes / (ms * 1e-3) / 1e9 / hbm_peak, valid_frac=float(out[1].float().mean()),
                launches={k: float(np.median(v)) for k, v in per.items()})


def bench_ransac(ctx, ffma_peak, n=8700, B=16, H=4096, mode=ops.SCORE_BEARING):
    rng = np.random.default_rng(0)
    cap = 16384
    p_cur = rng.normal(size=(B, cap, 3)).astype(np.float32) * 2
    ang = 0.02
    R = np.array([[np.cos(ang), -np.sin(ang), 0], [np.sin(ang), np.cos(ang), 0], [0, 0, 1]], np.float32)
    p_ref = p_cur @ R.T + np.float32([0.03, 0.01, -0.02]) + rng.normal(0, 0.01, p_cur.shape).astype(np.float32)
    p_ref[:, ::3] = rng.normal(size=p_ref[:, ::3].shape).astype(np.float32) * 2
    f = p_cur / np.linalg.norm(p_cur, axis=2, keepdims=True)
    cam = np.zeros((B, cap), np.uint8)
    cam[:, n // 2:] = 1
    rig = np.zeros((2, 3, 4)); rig[:, :, :3] = np.eye(3); rig[0, 2, 3] = 0.12
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    hyp = d(rng.integers(0, 2 ** 32, (H, 3), dtype=np.uint64).astype(np.uint32).view(np.int32))
    args = (d(p_ref), d(p_cur), torch.full((B,), n, dtype=torch.int32, device="cuda"), hyp, mode,
            1.0 - np.cos(np.deg2rad(5.0)) if mode == ops.SCORE_BEARING else 0.05)
    kw = dict(f_cur=d(f.astype(np.float32)), cam=d(cam), rig=rig, n_cams=2)
    ms = timeit(lambda: ctx.ransac_p3d(*args, **kw), iters=10)
    pairs = float(B) * n * H
    fl = pairs * (45.0 if mode == ops.SCORE_BEARING else 30.0)
    return dict(kernel="ransac(all 4 kernels)", mode=int(mode), ms=ms, pairs_per_s=pairs / (ms * 1e-3),
                tflops=fl / (ms * 1e-3) / 1e12, frac_of_ffma_peak=fl / (ms * 1e-3) / 1e12 / ffma_peak)


def bench_remap(ctx, hbm_peak, B=16, H=2048, W=2048, rows=849, cols=2400, offset=False):
    """offset: the sources start one byte into their buffers, so the generic remap_kernel<3> runs instead of remap3b_kernel
    (which needs a 4-byte aligned source with src_w % 4 == 0)."""
    g = torch.Generator(device="cuda").manual_seed(2)
    n, o = B * H * W * 3, int(offset)
    srcs = [torch.randint(0, 256, (n + o,), dtype=torch.uint8, device="cuda", generator=g)[o:].view(B, H, W, 3) for _ in range(2)]
    # annular LUTs like the real ones: pano (r, c) -> circle of radius growing with r
    r = torch.arange(rows, device="cuda", dtype=torch.float64)[:, None]
    c = torch.arange(cols, device="cuda", dtype=torch.float64)[None, :]
    luts = []
    for lo, hi in ((0.13 * H, 0.47 * H), (0.03 * H, 0.12 * H)):
        rad = lo + (hi - lo) * r / rows
        ang = 2 * np.pi * (1 - c / cols)
        mx = (W / 2 + rad * torch.cos(ang)).contiguous()
        my = (H / 2 + rad * torch.sin(ang)).contiguous()
        luts.append(ctx.lut_pack(mx, my, (H, W)))
    lut = torch.stack(luts).contiguous()
    out = ctx.remap(srcs[0], lut)
    it = [0]

    def run():
        ctx.remap(srcs[it[0] & 1], lut, out=out)
        it[0] += 1
    ms = timeit(run)
    alg = B * (2 * rows * cols * (8 + 3) + H * W * 3)
    dram = B * (2 * rows * cols * 3 + H * W * 3)
    return dict(kernel="remap", src_w=W, src_offset=o, ms=ms, gbps_algorithmic=alg / (ms * 1e-3) / 1e9,
                frac_of_hbm_peak=alg / (ms * 1e-3) / 1e9 / hbm_peak, gbps_src_plus_dst=dram / (ms * 1e-3) / 1e9)


def bench_rgbd(ctx, hbm_peak, B=256, h=480, w=640, n=1000):
    """RGB-D comparison path (BASELINE config 5, SURVEY 8a F12): radial depth -> Z over whole 640 x 480 maps (4 B in, 4 B out
    per pixel) and back-projection + range gate at n keypoints per frame (gather: 4 B depth + 8 B index in, 25 B out)."""
    g = torch.Generator(device="cuda").manual_seed(7)
    cam = [525.0, 525.0, 319.5, 239.5, 1.0 / 1000.0, 0.0]                # fx, fy, cx, cy, focal_m, depth_is_Z = 0 (radial)
    depth = [torch.rand((B, h, w), device="cuda", generator=g) * 6.0 + 0.5 for _ in range(2)]
    u = torch.randint(0, w, (B, n), dtype=torch.int32, device="cuda", generator=g)
    v = torch.randint(0, h, (B, n), dtype=torch.int32, device="cuda", generator=g)
    it = [0]

    def run_z():
        ctx.rgbd_depth_to_z(cam, depth[it[0] & 1])
        it[0] += 1

    def run_bp():
        ctx.rgbd_backproject(cam, depth[it[0] & 1], u, v, 0.8, 7.0)
        it[0] += 1
    ms_z, ms_bp = timeit(run_z), timeit(run_bp)
    gbps = B * h * w * 8 / (ms_z * 1e-3) / 1e9
    return dict(kernel="rgbd", frames=B, ms_depth_to_z=ms_z, gbps_depth_to_z=gbps, frac_of_hbm_peak=gbps / hbm_peak,
                ms_backproject=ms_bp, keypoints_per_s=B * n / (ms_bp * 1e-3), frames_per_s_both=B / ((ms_z + ms_bp) * 1e-3))


def card():
    """The card's name and power limit, read in the same run as the numbers they qualify."""
    import subprocess
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return dict(gpu=torch.cuda.get_device_name(0), power_limit=pl)


def bench_l2(ctx, dim, sizes, engine):
    """Both float-descriptor L2 engines on the same segment shapes: "int" = sos_l2_top2 on integer-valued SIFT-like rows,
    "float" = sos_l2f_top2 on RootSIFT-like rows (non-integer).  Executed bf16 FLOP/s counts the padded tiles and the MMA
    instructions each engine issues (9 x K16 per tile pair, resp. 3 ceil(dim / 16) + 1)."""
    rng = np.random.default_rng(dim)
    nq = np.array([a for a, _ in sizes], np.int32)
    nt = np.array([b for _, b in sizes], np.int32)
    h = rng.gamma(0.7, 28.0, (int(nq.sum() + nt.sum()), dim))
    if engine == "int":
        x = np.clip(h, 0, 255).round().astype(np.float32)
    else:
        x = np.sqrt(h / h.sum(1, keepdims=True)).astype(np.float32)
    tq, tt = x[:nq.sum()], x[nq.sum():]
    q_start = np.concatenate([[0], np.cumsum(nq)[:-1]]).astype(np.int32)
    t_start = np.concatenate([[0], np.cumsum(nt)[:-1]]).astype(np.int32)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    args = (d(tq), d(tt), d(q_start), d(nq), d(t_start), d(nt), int(nq.max()), int(nt.max()))
    stats = torch.zeros(ops.L2F_STATS, dtype=torch.int32, device="cuda")
    fn = (lambda: ctx.l2_top2(*args)) if engine == "int" else (lambda: ctx.l2f_top2(*args, stats=stats))
    ms = timeit(fn, iters=20)
    n_mma = 9 if engine == "int" else 3 * -(-dim // 16) + 1
    flops = sum(2.0 * (-(-a // 256) * 256) * (-(-b // 128) * 128) * 16 * n_mma for a, b in sizes)
    r = dict(kernel="l2_top2" if engine == "int" else "l2f_top2", dim=dim, segments=len(sizes),
             shape=f"{sizes[0][0]}x{sizes[0][1]}" if len(set(sizes)) == 1 else "mixed", ms=ms,
             bf16_tflops_executed=flops / (ms * 1e-3) / 1e12)
    if engine == "float":
        r["redecided_share"] = int(stats[ops.L2F_STAT_REDECIDED]) / int(nq.sum())
        r["band_ratio_max"] = int(stats[ops.L2F_STAT_BAND_PPM]) * 1e-6
    return r


def bench_l2_real(ctx):
    """Re-decided share of sos_l2f_top2 on live cv2 KAZE and RootSIFT descriptors of a seeded synthetic frame pair."""
    import cv2
    rng = np.random.default_rng(21)
    img = cv2.GaussianBlur((rng.random((960, 1280)) * 255).astype(np.uint8), (0, 0), 2.0)
    for _ in range(200):
        c = tuple(int(v) for v in rng.integers(0, [1280, 960]))
        cv2.circle(img, c, int(rng.integers(4, 40)), int(rng.integers(0, 255)), -1)
    rot = cv2.warpAffine(img, cv2.getRotationMatrix2D((640, 480), 12.0, 1.05), (1280, 960))
    sift = cv2.SIFT_create(nfeatures=8000)
    root = lambda v: np.sqrt(v / np.maximum(v.sum(1, keepdims=True), 1e-12)).astype(np.float32)
    out = []
    for name, det, post in (("KAZE", cv2.KAZE_create(), lambda v: v), ("RootSIFT", sift, root)):
        q, t = post(det.detectAndCompute(img, None)[1]), post(det.detectAndCompute(rot, None)[1])
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        z = d(np.zeros(1, np.int32))
        stats = torch.zeros(ops.L2F_STATS, dtype=torch.int32, device="cuda")
        args = (d(q), d(t), z, d(np.array([len(q)], np.int32)), z, d(np.array([len(t)], np.int32)), len(q), len(t))
        ms = timeit(lambda: ctx.l2f_top2(*args, stats=stats), iters=10)
        out.append(dict(kernel="l2f_top2", descriptors=name, dim=q.shape[1], nq=len(q), nt=len(t), ms=ms,
                        redecided_share=int(stats[ops.L2F_STAT_REDECIDED]) / len(q),
                        band_ratio_max=int(stats[ops.L2F_STAT_BAND_PPM]) * 1e-6))
    return out


def main():
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    ctx = ops.Context(0)
    res = []
    if what in ("hamming", "all"):
        pk = ctx.peak_popc()
        res.append(bench_hamming(ctx, pk, top2=False))
        res.append(bench_hamming(ctx, pk, top2=True))
        res.append(dict(bench_hamming(ctx, pk, n=667, segs=192, top2=False), note="stereo-like 192 x 667^2"))
    if what in ("ransac", "all"):
        pk = ctx.peak_ffma()
        res.append(bench_ransac(ctx, pk))
        res.append(bench_ransac(ctx, pk, mode=ops.SCORE_EUCLID))
    if what in ("remap", "all"):
        res.append(bench_remap(ctx, 6451.2))
        res.append(bench_remap(ctx, 6451.2, offset=True))
        res.append(bench_remap(ctx, 6451.2, W=2046))   # rows not a multiple of 4 bytes: generic kernel from an aligned source
    if what in ("dense", "all"):
        res.append(bench_dense(ctx, 6451.2))
    if what in ("rgbd", "all"):
        res.append(bench_rgbd(ctx, 6451.2))
    if what == "l2":
        res.append(card())
        stereo = [(700 - 5 * s, 700 + 5 * s) for s in range(12)]
        for dim in (64, 128):
            for sizes in (stereo, [(8000, 8000)]):
                res.append(bench_l2(ctx, dim, sizes, "int"))
                res.append(bench_l2(ctx, dim, sizes, "float"))
        res.extend(bench_l2_real(ctx))
    for r in res:
        print(json.dumps(r))


if __name__ == "__main__":
    main()
