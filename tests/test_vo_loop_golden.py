"""CPU: oracle/driver.py (the restatement of the reference's VO loop) against the reference's OWN run_VO
(pose_est_tools.py:1264-1678), which oracle/gen_vo_golden.py drove unmodified over a rendered 9-frame sequence with a
pyopengv stub backed by oracle/p3p.py + oracle/ransac.py.  Fed the features the reference detected, the restated loop must
produce the same keyframe ids and the same estimated_frame_poses_TUM.txt."""
import numpy as np

from oracle import driver as odriver, hamming, p3p, pipeline, ransac
from vo_single_camera_sos_b200 import synth

import _vo_golden


def oracle_track_fn(g):
    """TrackerStereoSE3.track_frame (pose_est_tools.py:736-847) with the reference's argument list for OpenGV: temporal matching
    of both views, stacking, RANSAC over the seeded list (bearings + reference 3D points only), LM refinement on the inliers."""
    rig, hyp, thr = _vo_golden.rig_matrix(g), _vo_golden.hypothesis_list(g), float(g["threshold"])
    max_du = float(g["max_horizontal_diff_f2f"])

    calls = []

    def track(ref, cur):
        parts = []
        for view, (uvk, dk, bk) in enumerate((("uv_top", "desc_top", "b_top"), ("uv_bot", "desc_bot", "b_bot"))):
            if len(cur[dk]) == 0 or len(ref[dk]) == 0:
                continue
            qi, ti = pipeline._bf_sorted(cur[dk], ref[dk])
            ok = hamming.filter_pixel_correspondences(ref[uvk][ti], cur[uvk][qi], -1, max_du)
            qi, ti = qi[ok], ti[ok]
            parts.append((ref["xyz"][ti], cur[bk][qi], np.full(len(qi), view, np.uint8)))
        if not parts:
            return None
        p_ref, f_cur, cam = (np.concatenate(x) for x in zip(*parts))
        p32, f32 = p_ref.astype(np.float32), f_cur.astype(np.float32)
        M, h, c, inl, _ = p3p.ransac_p3p(p32, f32, cam, rig, hyp, thr)
        calls.append(dict(points=p_ref, bearings=f_cur, cam=cam, best_hyp=h, inliers=np.nonzero(inl)[0]))
        out = dict(n_corr=len(p_ref), best_hyp=h, best_count=c)
        if h >= 0:
            idx = np.nonzero(inl)[0]
            out["refit"] = ransac.refine_pose_lm(p32[idx], f32[idx], np.asarray(M, np.float64).astype(np.float32), cam[idx], rig)[0]
        return out
    track.calls = calls
    return track


def test_restated_vo_loop_reproduces_the_reference_run():
    g, frames = _vo_golden.load()
    n = len(frames)
    rig = synth.make_rig(int(g["width"]), int(g["height"]), int(g["pano_cols"]), seed=int(g["seed"]))
    assert np.allclose(np.asarray(g["cam_offsets"])[0], rig.f_top) and np.allclose(np.asarray(g["cam_offsets"])[1], rig.f_bot)
    cap = 4096
    pano_g = _vo_golden.pano_geometry(g)
    assert pano_g == _vo_golden.pano_geometry(g, "bot")          # both mirrors share the panorama grid (camera_models.py:2795-2800)
    frame_fn = lambda f: pipeline.stereo_frame(pano_g, rig.f_top, rig.f_bot, f["px_top"], f["desc_top"], f["boff_top"],
                                               f["px_bot"], f["desc_bot"], f["boff_bot"], cap=cap)
    track_fn = oracle_track_fn(g)
    out = odriver.run_vo(frames, frame_fn=frame_fn, track_fn=track_fn)
    assert out["status"] == "ok"
    # what the restated front half (stereo matching, lifting, triangulation, range gate, temporal matching, stacking) hands to
    # RANSAC for every frame, against what the reference's tracker handed to its pyopengv call: same correspondences in the
    # same order (float64 values to 1e-9), hence the same winner and the same inlier indices
    assert len(track_fn.calls) == n - 1
    for i, c in enumerate(track_fn.calls, start=1):
        assert c["points"].shape == g[f"f{i}_ransac_points"].shape, i
        assert np.array_equal(c["cam"], g[f"f{i}_ransac_cam"])
        assert np.allclose(c["points"], g[f"f{i}_ransac_points"], rtol=0, atol=1e-9), i
        assert np.allclose(c["bearings"], g[f"f{i}_ransac_bearings"], rtol=0, atol=1e-12), i
        assert c["best_hyp"] == int(g[f"f{i}_ransac_best_hyp"]) and np.array_equal(c["inliers"], g[f"f{i}_ransac_inliers"]), i
    assert out["keyframe_ids"] == g["keyframe_ids"].tolist()
    assert 1 < len(out["keyframe_ids"]) < n          # the golden exercises both branches of the keyframe decision
    est = g["est_tum"]
    T_ref = [_vo_golden.tum_to_matrix(est[i]) for i in range(n)]
    # per frame: pose relative to its tracking reference (the keyframe current when the frame was tracked) to 2e-7 — the TUM file
    # prints float64 repr, the inputs of RANSAC agree to 1e-9 (checked above), and the Levenberg-Marquardt minimiser is a
    # function of them; the absolute poses chain up to 8 such links: 2e-6
    parent = 0
    for i in range(1, n):
        rel_ref = np.linalg.inv(T_ref[parent]) @ T_ref[i]
        rel_got = np.linalg.inv(out["poses_wrt_S"][parent]) @ out["poses_wrt_S"][i]
        assert np.allclose(rel_got, out["poses_wrt_keyframe"][i], atol=1e-12)
        assert np.allclose(rel_got, rel_ref, atol=2e-7), (i, np.abs(rel_got - rel_ref).max())
        assert np.allclose(out["poses_wrt_S"][i], T_ref[i], atol=2e-6), i
        if i in out["keyframe_ids"]:
            parent = i
    # the TUM writer: same text as the reference's file (pose_est_tools.py:1609-1612) wherever the poses agree to the last bit
    ref_lines = bytes(g["est_tum_text"]).decode().strip().split("\n")
    assert len(ref_lines) == n and ref_lines[0] == odriver.tum_line(0, out["poses_wrt_S"][0])   # identical text for frame 0
    for i, line in enumerate(ref_lines):
        a = np.array(line.split()[1:], float)
        b = np.array(odriver.tum_line(i, out["poses_wrt_S"][i]).split()[1:], float)
        assert line.split()[0] == str(i) and np.allclose(a, b, atol=2e-6)
