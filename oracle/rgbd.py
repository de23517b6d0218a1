"""CPU restatement of one RGB-D frame / frame pair and of the RGB-D VO loop, chaining the oracle stages the way the
reference's RGBDFrame.establish_keypoints (pose_est_tools.py:600-623) and TrackerRGBDSE3.track_frame
(pose_est_tools.py:880-958) chain them, and run_VO (pose_est_tools.py:1403-1628) with one camera.  TEST INFRASTRUCTURE
ONLY (see oracle/__init__.py): the checker of the RGB-D front-end (sos_frontend_create_rgbd) and of the batched driver
on it, and the CPU arm of scripts/bench_rgbd.py."""
from __future__ import annotations

import numpy as np

from . import driver, geometry, hamming, p3p, pipeline, ransac


def rgbd_frame(cam, depth, px, desc, min_z=0.8, max_z=7.0):
    """RGBDFrame.establish_keypoints (pose_est_tools.py:600-623) on given keypoints: pixel (trunc(x), trunc(y))
    (astype(np.uint), :612), geometry.rgbd_backproject and its |Z| gate, then kpts[valid] in row order.  A keypoint whose
    truncated pixel lies outside the map is dropped (the reference would raise on it).  cam: dict over
    geometry.RGBD_FIELDS; px float32 [n,2]; desc uint8 [n,32]."""
    px = np.asarray(px, np.float32).reshape(-1, 2)
    h, w = depth.shape
    tx, ty = np.trunc(px[:, 0]), np.trunc(px[:, 1])
    with np.errstate(invalid="ignore"):
        inside = (tx >= 0) & (tx < w) & (ty >= 0) & (ty < h)
    u = np.where(inside, tx, 0).astype(np.int64)
    v = np.where(inside, ty, 0).astype(np.int64)
    xyz, bearing, valid = geometry.rgbd_backproject(cam, depth, u, v, min_z, max_z)
    valid &= inside
    return dict(uv=px[valid], xyz=xyz[valid], b=bearing[valid], desc=np.asarray(desc)[valid], src=np.flatnonzero(valid))


def rgbd_track_pair(ref, cur, hyp, threshold, max_du, solver="arun", refine="lm", pts=None):
    """TrackerRGBDSE3.track_frame (pose_est_tools.py:880-958) on two rgbd_frame results: 1-NN matching query = current,
    train = reference, sorted by distance, |du| gate; RANSAC with a central camera and the bearing score on the float32
    points (Arun hypotheses, or with solver="p3p" the three-point solver on hyp [n_hyp,4]); then refine ("lm", "arun",
    "none").  pts(frame) -> (xyz, bearing) replaces the frame's own float64 points (e.g. by the device's float32 ones).
    Returns None when either frame has no keypoints."""
    if len(cur["desc"]) == 0 or len(ref["desc"]) == 0:
        return None
    qi, ti = pipeline._bf_sorted(cur["desc"], ref["desc"])
    ok = hamming.filter_pixel_correspondences(ref["uv"][ti], cur["uv"][qi], -1, max_du)
    qi, ti = qi[ok], ti[ok]
    (xr, _), (xc, bc) = (pts(ref), pts(cur)) if pts is not None else ((ref["xyz"], ref["b"]), (cur["xyz"], cur["b"]))
    f32 = lambda a: np.asarray(a, np.float32)
    p_ref, p_cur, f_cur = f32(xr[ti]), f32(xc[qi]), f32(bc[qi])
    if solver == "p3p":
        pose, best, count, mask, counts = p3p.ransac_p3p(p_ref, f_cur, None, None, hyp, threshold)
        o = dict(pose=pose if pose is not None else np.full((3, 4), np.nan), best_hyp=best, best_count=count, mask=mask,
                 counts=counts)
    else:
        o = ransac.ransac_p3d(p_ref, p_cur, hyp, "bearing", threshold, f_cur=f_cur)
    if o["best_hyp"] >= 0:
        if refine == "lm":   # absolute_pose_optimize_nonlinear on the inliers, started at the RANSAC pose (:937)
            o["refit"] = ransac.refine_pose_lm(p_ref, f_cur, o["pose"], mask=o["mask"])[0]
        elif refine == "arun":
            o["refit"] = ransac.refit(p_ref, p_cur, o["mask"])
        else:
            o["refit"] = o["pose"]
    o["n_corr"] = len(p_ref)
    o["pairs"] = (qi, ti)
    return o


def run_vo(frames, cam, hyp, threshold, max_du, thresholds=None, refine="lm", solver="arun", min_correspondences=6,
           units_to_m=1.0):
    """oracle.driver.run_vo over rgbd_frame / rgbd_track_pair with number_of_cams = 1.  frames: dicts with depth, px, desc
    of ONE frame each (trimmed to their keypoints).  TrackerRGBDSE3.track_frame refuses fewer than 2 * 3 * 1
    correspondences (min_correspondences): such a pair is a tracking failure."""
    def track(ref, cur):
        o = rgbd_track_pair(ref, cur, hyp, threshold, max_du, solver=solver, refine=refine)
        return None if o is None or o["n_corr"] < min_correspondences else o
    return driver.run_vo(frames, thresholds=thresholds, units_to_m=units_to_m, number_of_cams=1,
                         frame_fn=lambda f: rgbd_frame(cam, f["depth"], f["px"], f["desc"]), track_fn=track)
