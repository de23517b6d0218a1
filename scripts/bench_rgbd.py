#!/usr/bin/env python
"""BASELINE configuration 5 (RGB-D comparison path, demo_vo_rgbd.py) on one GPU: 640x480 depth maps, 2 000 keypoints per
frame, both depth encodings, make_rgbd_sequence frames.  Paths timed in one run, their steps alternating:
  graph   Frontend.step_rgbd on device-resident inputs (captured CUDA graph), steps queued back to back
  host    Frontend.submit_host_rgbd / wait_host from pinned memory (two steps in flight), and an H2D-only probe of the same
          bytes with the same copy sizes
  mirror  the per-pair Python path: RGBDFrame + TrackerRGBDSE3.track_frame on the same frames (one frame pair per call)
  oracle  the CPU composition oracle.rgbd.rgbd_frame + rgbd_track_pair (NumPy / OpenCV)
The GPU paths run blocks of 10 consecutive steps each, alternating block by block (medians over the blocks); plus
per-kernel times (profile_begin / profile_end, a run of its own), launches and H2D bytes per step, and the card's name
and power limit.
python scripts/bench_rgbd.py [--batch 32 128] [--steps 50] [--out file.json]"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vo_single_camera_sos_b200 import ops, pyopengv, synth  # noqa: E402
from vo_single_camera_sos_b200.frontend import Frontend, RgbdFrontendConfig  # noqa: E402

N_KP = 2000
THR = 1.0 - math.cos(math.radians(5.0))


def card():
    """The card's name and power limit, read in the same run as the numbers they qualify."""
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return dict(gpu=torch.cuda.get_device_name(0), power_limit=pl)


def by_name(launches):
    agg = {}
    for name, t in launches:
        k = name.split("#")[0].split(":")[0]
        agg[k] = agg.get(k, 0.0) + t
    return {k: round(v, 4) for k, v in sorted(agg.items(), key=lambda kv: -kv[1])}


def median_ms(xs):
    return round(float(np.median(xs)) * 1e3, 4)


def run_config(ctx, B, depth_is_Z, steps, pair_samples):
    seq = synth.make_rgbd_sequence(2 * B + 1, N_KP, depth_is_Z, seed=11)
    batches = [seq.inputs(range(k * B, (k + 1) * B), N_KP) for k in range(2)]
    hyp = pyopengv.hypothesis_list(210, 0)
    hyp_d = torch.from_numpy(hyp.view(np.int32)).cuda()
    cfg = RgbdFrontendConfig(batch=B, cam=seq.cam_vector(), max_kp=N_KP, refine_iters=60)
    fg, fh = Frontend(ctx, cfg, None, hyp_d), Frontend(ctx, cfg, None, hyp_d)
    dev = [[torch.from_numpy(np.ascontiguousarray(bt[k])).cuda() for k in ("depth", "px", "desc", "n_kp")] for bt in batches]
    pinned = [[torch.from_numpy(np.ascontiguousarray(bt[k])).pin_memory() for k in ("depth", "px", "desc", "n_kp")]
              for bt in batches]
    h2d_bytes, _ = fh.host_bytes()
    staging = [torch.empty(p.numel() * p.element_size(), dtype=torch.uint8, device="cuda") for p in pinned[0]]
    copy_stream = torch.cuda.Stream()

    # each path runs `block` consecutive steps as a user would (graph launches queued back to back, host steps two in
    # flight), timed to the end of its last step; the paths alternate block by block
    def graph_block(k0):
        for k in range(k0, k0 + block):
            fg.step_rgbd(*dev[k & 1])
        torch.cuda.synchronize()

    def host_block(k0):
        tickets = []
        for k in range(k0, k0 + block):
            tickets.append(fh.submit_host_rgbd(*pinned[k & 1]))
            if len(tickets) > 1:
                fh.wait_host(tickets.pop(0))
        while tickets:
            fh.wait_host(tickets.pop(0))

    def h2d_block(k0):
        with torch.cuda.stream(copy_stream):
            for k in range(k0, k0 + block):
                for s, p in zip(staging, pinned[k & 1]):
                    s.copy_(p.view(-1).view(torch.uint8), non_blocking=True)
        copy_stream.synchronize()

    block = 10
    paths = (("graph", graph_block), ("host", host_block), ("h2d", h2d_block))
    for _, fn in paths:   # warm-up: graph capture, staging, first launches
        fn(0)
    t = {name: [] for name, _ in paths}
    for r in range(max(1, steps // block)):
        for name, fn in paths:
            t0 = time.perf_counter()
            fn(r * block)
            t[name].append((time.perf_counter() - t0) / block)
    launches = fg.buffers()["launches_per_step"]
    stats = fg.buffers()["stats"].cpu().numpy()
    # per-kernel times: eager launches under events, a run of its own
    fg.profile_begin()
    for k in range(3):
        fg.step_rgbd(*dev[k & 1])
    torch.cuda.synchronize()
    prof = fg.profile_end()
    kernels = {k: round(v / 3.0, 4) for k, v in by_name(prof).items()}
    # the per-pair mirror and the CPU oracle on the first pair_samples pairs of the same frames
    from omnistereo import pose_est_tools
    from omnistereo.camera_models import RGBDCamModel
    from oracle import geometry, rgbd as orgbd
    c = seq.cam
    cam = RGBDCamModel(fx=c["fx"], fy=c["fy"], center_x=c["center_x"], center_y=c["center_y"], depth_is_Z=depth_is_Z, units="m")
    tracker = pose_est_tools.TrackerRGBDSE3(cam)
    rgb = np.zeros((480, 640, 3), np.uint8)
    camd = dict(zip(geometry.RGBD_FIELDS, seq.cam_vector()))
    t_mirror, t_oracle = [], []
    prev_m = prev_o = None
    for i in range(pair_samples + 1):
        f = seq.frames[i]
        t0 = time.perf_counter()
        kp = [cv2.KeyPoint(float(x), float(y), 7.0) for x, y in f["px"]]
        fm = pose_est_tools.RGBDFrame(cam, rgb, f["depth"], i, features=(kp, f["desc"]))
        if prev_m is not None:
            tracker.track_frame(prev_m, fm)
        t1 = time.perf_counter()
        fo = orgbd.rgbd_frame(camd, f["depth"], f["px"], f["desc"])
        if prev_o is not None:
            orgbd.rgbd_track_pair(prev_o, fo, hyp, THR, 319.5, refine="lm")
        t2 = time.perf_counter()
        if i > 0:
            t_mirror.append(t1 - t0)
            t_oracle.append(t2 - t1)
        prev_m, prev_o = fm, fo
    fg.close()
    fh.close()
    g, h = median_ms(t["graph"]), median_ms(t["host"])
    return dict(
        batch=B, depth_is_Z=bool(depth_is_Z), keypoints_per_frame=N_KP, steps=steps,
        graph_ms_per_step=g, graph_frame_pairs_per_s=round(B / (g * 1e-3), 1),
        host_ms_per_step=h, host_frame_pairs_per_s=round(B / (h * 1e-3), 1),
        h2d_probe_ms_per_step=median_ms(t["h2d"]), h2d_bytes_per_step=int(h2d_bytes),
        mirror_ms_per_pair=median_ms(t_mirror), oracle_ms_per_pair=median_ms(t_oracle), pair_samples=pair_samples,
        launches_per_step=int(launches), kernel_ms_per_step=kernels, kernel_ms_total=round(sum(kernels.values()), 4),
        mean_valid_keypoints=float(stats[:, 0].mean()), mean_correspondences=float(stats[:, 1].mean()),
        mean_inliers=float(stats[:, 2].mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, nargs="+", default=[32, 128])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--pairs", type=int, default=8, help="frame pairs timed on the mirror and oracle paths")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_rgbd.py needs a CUDA device")
    ctx = ops.Context(0)
    out = dict(card(), workload="config 5: 640x480 depth, 2000 keypoints per frame, make_rgbd_sequence(seed=11)", results=[])
    for B in args.batch:
        for depth_is_Z in (True, False):
            r = run_config(ctx, B, depth_is_Z, args.steps, args.pairs)
            print(json.dumps(r), flush=True)
            out["results"].append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
