#!/usr/bin/env python
"""Image-in throughput of the whole front-end on one GPU (SURVEY §8f N3 + the hot path): rendered omni images -> panoramas,
features, matching, triangulation, RANSAC poses.  Three paths in one run, their steps alternating:
  python  features.step_images: the Python composition of the feature-front calls, then Frontend.step
  graph   Frontend.step_images: detection inside the step's CUDA graph, omni images resident in HBM
  host    Frontend.submit_host_images / wait_host: pinned host images in, poses out (band uploads, two steps in flight)
python scripts/bench_images.py [--workload c2] [--batch 16 32] [--steps 20] [--out file.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch
import torch.nn.functional as Fn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vo_single_camera_sos_b200 import ops, workload  # noqa: E402
from vo_single_camera_sos_b200.features import FeatureFront, azimuthal_masks, step_images  # noqa: E402


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
    return {k: round(v, 3) for k, v in agg.items()}


def candidate_counts(ctx, pano, masks, median):
    """Shi-Tomasi candidates (local maxima above quality 0.01 of the mask's maximum) of every (frame, view, mask) list of
    one step: what the selection has to rank, and what sizes its shared memory."""
    B = pano.shape[0]
    imgs = pano.reshape(B * 2, *pano.shape[2:])
    if median:
        imgs = ctx.median_blur_11(imgs)
    gray = ctx.bgr_to_gray(imgs).reshape(B, 2, *pano.shape[2:4])
    out = []
    for view in range(2):
        eig = ctx.corner_min_eigenval(gray[:, view].contiguous())                     # [B, H, W]
        peak = Fn.max_pool2d(eig[:, None], 3, 1, 1)[:, 0]
        inner = torch.zeros_like(eig, dtype=torch.bool)
        inner[:, 1:-1, 1:-1] = True
        for m in masks[view]:
            mb = m.bool()
            mx = torch.where(mb, eig, torch.zeros_like(eig)).amax(dim=(1, 2))
            thr = (mx.double() * 0.01).float()
            cand = inner & mb & (eig > thr[:, None, None]) & (eig == peak) & (eig > 0)
            out += cand.sum(dim=(1, 2)).tolist()
    return np.array(out)


def run(a, B):
    ctx = ops.Context(0)
    w = workload.build(ctx, a.workload, batch=B, n_frames=2 * B + 1, seed=0, score_mode=ops.SCORE_BEARING)
    c = workload.CONFIGS[a.workload]
    rows, cols = w.cfg.pano_rows, w.cfg.pano_cols
    N = min(w.cfg.max_feat_per_bucket, c["feat"] // 12 + 1)
    valid = ((w.lut >> 48) & 0xF) != 0
    masks = []
    for view in range(2):
        v = cv2.erode(valid[view].cpu().numpy().astype(np.uint8), np.ones((7, 7), np.uint8)).astype(bool)
        masks.append(azimuthal_masks(rows, cols, 12) & (v[None] * 255).astype(np.uint8))
    front = FeatureFront(ctx, masks[0], masks[1], corners_per_bucket=N, max_feat_per_view=w.cfg.max_feat_per_view)
    renderer = workload.DeviceRenderer(ctx, w)
    sets = [torch.stack([renderer.render(w.trajectory[s * B + i]) for i in range(B)]).contiguous() for s in range(2)]
    pinned = [s.cpu().pin_memory() for s in sets]
    fe_py, fe_graph, fe_host = w.frontend(ctx), w.frontend(ctx), w.frontend(ctx)
    for fe in (fe_graph, fe_host):
        fe.set_detector(masks[0], masks[1], N)
    # warm-up (captures the graphs, sizes the arenas); the python and graph front-ends see the same frames in the same
    # order, so their poses must agree bit for bit
    for s in range(3):
        step_images(fe_py, front, sets[s % 2], w.lut)
        fe_graph.step_images(sets[s % 2])
        fe_host.step_host_images(pinned[s % 2])
    torch.cuda.synchronize()
    same = True
    t = {"python": 0.0, "graph": 0.0}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for s in range(a.steps):
        ev[0].record()
        step_images(fe_py, front, sets[s % 2], w.lut)
        ev[1].record()
        fe_graph.step_images(sets[s % 2])
        ev[2].record()
        torch.cuda.synchronize()
        t["python"] += ev[0].elapsed_time(ev[1])
        t["graph"] += ev[1].elapsed_time(ev[2])
        same &= torch.equal(fe_py.buffers()["pose"], fe_graph.buffers()["pose"]) and \
            torch.equal(fe_py.buffers()["stats"], fe_graph.buffers()["stats"])
    # host path, end to end: two steps in flight, wall clock from the first submit to the last wait
    t0 = time.perf_counter()
    tickets = []
    for s in range(a.steps):
        tickets.append(fe_host.submit_host_images(pinned[s % 2]))
        if len(tickets) == 2:
            fe_host.wait_host(tickets.pop(0))
    for tk in tickets:
        fe_host.wait_host(tk)
    host_ms = (time.perf_counter() - t0) * 1e3 / a.steps
    # device time of every launch inside one step (profiled steps run eagerly)
    # (python: the feature-front calls only; the front-end's own launches are timed on its private context, whose
    # profile would also count the host's wait inside sos_gft_detect)
    ctx.profile_begin()
    step_images(fe_py, front, sets[0], w.lut)
    py_launches = ctx.profile_end()
    fe_graph.profile_begin()
    fe_graph.step_images(sets[0])
    graph_launches = fe_graph.profile_end()
    counts = candidate_counts(ctx, fe_graph.buffers()["pano"], [torch.from_numpy(m).to(ctx.device) for m in masks], True)
    st = fe_graph.buffers()["stats"].cpu().numpy()
    ds = fe_graph.features()["detect_stats"].cpu().numpy()
    ms = {k: v / a.steps for k, v in t.items()}
    return {"metric": "image_in_frame_pairs_per_s", "workload": a.workload, "batch": B, "steps": a.steps, **card(),
            "python_ms_per_step": round(ms["python"], 3), "graph_ms_per_step": round(ms["graph"], 3),
            "host_ms_per_step": round(host_ms, 3),
            "python_frame_pairs_per_s": round(B / (ms["python"] * 1e-3), 1),
            "graph_frame_pairs_per_s": round(B / (ms["graph"] * 1e-3), 1),
            "host_frame_pairs_per_s": round(B / (host_ms * 1e-3), 1),
            "host_h2d_bytes_per_step": fe_host.host_images_bytes(),
            "graph_poses_equal_python": bool(same),
            "python_feature_front_ms_by_launch": by_name(py_launches),
            "python_feature_front_ms": round(sum(x for _, x in py_launches), 3),
            "graph_library_ms_by_launch": by_name(graph_launches),
            "graph_library_ms": round(sum(x for _, x in graph_launches), 3),
            "graph_launches_per_step": len(graph_launches), "corners_per_bucket": N,
            "candidates_per_list": {"lists": int(counts.size), "min": int(counts.min()), "p50": int(np.percentile(counts, 50)),
                                    "p90": int(np.percentile(counts, 90)), "p99": int(np.percentile(counts, 99)),
                                    "max": int(counts.max()), "over_1024": int((counts > 1024).sum()),
                                    "over_2048": int((counts > 2048).sum()), "over_4096": int((counts > 4096).sum()),
                                    "over_8192": int((counts > 8192).sum()), "over_16384": int((counts > 16384).sum())},
            "detect_stats_sum": ds.sum(axis=(0, 1)).tolist(),
            "stereo_correspondences": st[:, 0].tolist(), "temporal_correspondences": st[:, 1].tolist(),
            "ransac_inliers": st[:, 2].tolist()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--batch", type=int, nargs="+", default=[16])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the result lines to this JSON file")
    a = ap.parse_args()
    res = []
    for B in a.batch:
        r = run(a, B)
        print(json.dumps(r), flush=True)
        res.append(r)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
