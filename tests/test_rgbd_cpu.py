"""CPU: the synthetic RGB-D sequence (synth.make_rgbd_sequence), the RGB-D oracle composition (oracle.rgbd: rgbd_frame,
rgbd_track_pair, run_vo with one camera) and the driver's host logic for one camera."""
import math

import numpy as np
import pytest

from oracle import driver as odriver, geometry, rgbd as orgbd
from vo_single_camera_sos_b200 import synth
from vo_single_camera_sos_b200.pyopengv import hypothesis_list

THR = 1.0 - math.cos(math.radians(5.0))


@pytest.mark.parametrize("depth_is_Z", [True, False], ids=["Z", "radial"])
def test_sequence_depth_at_keypoints_and_determinism(depth_is_Z):
    s = synth.make_rgbd_sequence(4, 2000, depth_is_Z, seed=2)
    assert s.cam["fx"] == s.cam["fy"] == (525.0 if depth_is_Z else 554.256258)
    assert (s.cam["center_x"], s.cam["center_y"]) == (319.5, 239.5)
    for f in s.frames:
        assert f["depth"].shape == (480, 640) and f["depth"].dtype == np.float32
        assert f["px"].shape == (2000, 2) and f["px"].dtype == np.float32 and f["desc"].shape == (2000, 32)
        lm = f["landmark"] >= 0
        assert 0.7 < lm.mean() < 0.8                                    # about 25 % distractors
        ids = f["landmark"][lm]
        assert len(np.unique(ids)) == len(ids)
        u, v = np.trunc(f["px"][lm, 0]).astype(int), np.trunc(f["px"][lm, 1]).astype(int)
        assert len(np.unique(v * 640 + u)) == len(u)                    # one landmark per truncated pixel
    for i, f in enumerate(s.frames):
        lm = f["landmark"] >= 0
        P = (s.landmarks[f["landmark"][lm]] - s.trajectory[i][:3, 3]) @ s.trajectory[i][:3, :3]
        u, v = np.trunc(f["px"][lm, 0]).astype(int), np.trunc(f["px"][lm, 1]).astype(int)
        want = synth.rgbd_depth_value(s.cam, P[:, 2], u, v).astype(np.float32)
        assert np.array_equal(f["depth"][v, u], want)                   # the landmark's depth at its truncated pixel
        z = geometry.rgbd_depth_to_z(dict(zip(geometry.RGBD_FIELDS, s.cam_vector())), f["depth"])[v, u]
        np.testing.assert_allclose(z, P[:, 2], rtol=1e-6)
        mask = np.ones((480, 640), bool)
        mask[v, u] = False
        assert np.all(f["depth"][mask] == s.background)
    t = synth.make_rgbd_sequence(4, 2000, depth_is_Z, seed=2)
    for a, b in zip(s.frames, t.frames):
        for k in a:
            assert np.array_equal(a[k], b[k])
    other = synth.make_rgbd_sequence(4, 2000, depth_is_Z, seed=3)
    assert not np.array_equal(other.frames[1]["px"], s.frames[1]["px"])
    inp = s.inputs([1, 3], 2100)
    assert inp["n_kp"].tolist() == [2000, 2000] and np.array_equal(inp["px"][1, :2000], s.frames[3]["px"])
    assert not inp["px"][:, 2000:].any()


def test_rgbd_frame_drops_outside_pixels_and_compacts_in_order():
    s = synth.make_rgbd_sequence(1, 300, True, seed=4, background=3.0)
    f = s.frames[0]
    px, desc = f["px"].copy(), f["desc"]
    px[:5] = [[-3.5, 1.0], [640.0, 2.0], [3.0, 480.5], [np.nan, 1.0], [-0.5, -0.25]]
    cam = dict(zip(geometry.RGBD_FIELDS, s.cam_vector()))
    o = orgbd.rgbd_frame(cam, f["depth"], px, desc)
    assert not np.isin([0, 1, 2, 3], o["src"]).any() and 4 in o["src"]
    assert np.all(np.diff(o["src"]) > 0)
    keep = np.arange(5, 300)
    xyz, b, valid = geometry.rgbd_backproject(cam, f["depth"], np.trunc(px[keep, 0]).astype(int),
                                              np.trunc(px[keep, 1]).astype(int), 0.8, 7.0)
    assert np.array_equal(o["src"][1:], keep[valid])
    assert np.array_equal(o["xyz"][1:], xyz[valid]) and np.array_equal(o["b"][1:], b[valid])
    assert np.array_equal(o["desc"], desc[o["src"]]) and np.array_equal(o["uv"], px[o["src"]])


@pytest.mark.parametrize("depth_is_Z", [True, False], ids=["Z", "radial"])
def test_rgbd_track_pair_recovers_motion(depth_is_Z):
    s = synth.make_rgbd_sequence(2, 2000, depth_is_Z, seed=5)
    cam = dict(zip(geometry.RGBD_FIELDS, s.cam_vector()))
    fr = [orgbd.rgbd_frame(cam, f["depth"], f["px"], f["desc"]) for f in s.frames]
    o = orgbd.rgbd_track_pair(fr[0], fr[1], hypothesis_list(210, 0), THR, 319.5, refine="lm")
    qi, ti = o["pairs"]
    assert o["n_corr"] == len(qi) > 1000 and o["best_count"] > 400 and o["mask"].sum() == o["best_count"]
    assert np.all(np.abs(fr[1]["uv"][qi, 0] - fr[0]["uv"][ti, 0]) <= 319.5)
    T = np.linalg.inv(s.trajectory[0]) @ s.trajectory[1]
    assert np.allclose(o["pose"][:, :3], T[:3, :3], atol=5e-3) and np.allclose(o["pose"][:, 3], T[:3, 3], atol=2e-2)
    lid = [s.frames[i]["landmark"][fr[i]["src"]] for i in range(2)]
    assert np.mean(lid[1][qi][o["mask"]] == lid[0][ti][o["mask"]]) > 0.99      # the inliers are true correspondences
    assert np.all(np.isfinite(o["refit"]))
    assert orgbd.rgbd_track_pair(fr[0], dict(fr[1], desc=fr[1]["desc"][:0]), None, THR, 319.5) is None


def test_run_vo_refuses_fewer_than_six_correspondences():
    """TrackerRGBDSE3.track_frame refuses fewer than 2 * 3 * 1 correspondences: a frame with 5 keypoints fails the loop."""
    s = synth.make_rgbd_sequence(3, 600, True, seed=7)
    fr = [dict(depth=f["depth"], px=f["px"], desc=f["desc"]) for f in s.frames]
    cam = dict(zip(geometry.RGBD_FIELDS, s.cam_vector()))
    hyp = hypothesis_list(210, 0)
    ok = orgbd.run_vo(fr, cam, hyp, THR, 319.5, refine="none")
    assert ok["status"] == "ok" and len(ok["poses_wrt_S"]) == 3
    fr[2] = dict(fr[2], px=fr[2]["px"][:5], desc=fr[2]["desc"][:5])
    bad = orgbd.run_vo(fr, cam, hyp, THR, 319.5, refine="none")
    assert bad["status"] == "tracking failed at frame 2" and len(bad["poses_wrt_S"]) == 2
    assert orgbd.run_vo(fr, cam, hyp, THR, 319.5, refine="none", min_correspondences=2)["status"] == "ok"


def test_driver_layout_and_one_camera_bookkeeping():
    from vo_single_camera_sos_b200 import driver
    from vo_single_camera_sos_b200.frontend import FrontendConfig, RgbdFrontendConfig
    keys, shapes, cams, min_corr = driver.frontend_layout(RgbdFrontendConfig(batch=4, cam=[525, 525, 319.5, 239.5, 1e-3, 1]))
    assert keys == driver.RGBD_INPUT_KEYS == ("depth", "px", "desc", "n_kp") and cams == 1 and min_corr == 6
    assert shapes["depth"][0] == (4, 480, 640) and shapes["px"][0] == (4, 2000, 2) and shapes["n_kp"][0] == (4,)
    sos = FrontendConfig(batch=2, src_h=10, src_w=12, pano_rows=5, pano_cols=6, pano_top=[0] * 6, pano_bot=[0] * 6,
                         f_top=[0] * 3, f_bot=[0] * 3)
    keys, shapes, cams, min_corr = driver.frontend_layout(sos)
    assert keys == driver.INPUT_KEYS and cams == 2 and min_corr == 2 * 3 * (0.33 * 2)
    assert shapes["omni"][0] == (2, 10, 12, 3) and shapes["boff_top"][0] == (2, 13)
    c = RgbdFrontendConfig(batch=1, cam=[525, 526, 300.5, 239.5, 1e-3, 0]).to_c()
    assert c.temporal_max_du == 300.5 and c.refit == 2 and list(c.cam) == [525, 526, 300.5, 239.5, 1e-3, 0]
    # one camera: num_tracked = inliers (pose_est_tools.py:1513), against the sequential oracle on canned results
    rng = np.random.default_rng(1)
    steps = [np.eye(4)]
    for _ in range(30):
        T = np.eye(4)
        T[:3, 3] = rng.normal(size=3) * 0.01 + [0.012, 0, 0]
        steps.append(steps[-1] @ T)
    inl = rng.integers(20, 400, 31)
    frame_fn = lambda i: dict(idx=i, xyz=np.zeros((500, 3)))

    def track_fn(ref, cur):
        T = np.linalg.inv(steps[ref["idx"]]) @ steps[cur["idx"]]
        return dict(refit=T[:3], n_corr=int(inl[cur["idx"]]) + 5, best_hyp=0, best_count=int(inl[cur["idx"]]))
    th = dict(odriver.INDOOR, pos_min=0.03)
    want = odriver.run_vo(list(range(31)), thresholds=th, number_of_cams=1, frame_fn=frame_fn, track_fn=track_fn)
    st = driver.TrackingState(driver.KeyframePolicy(**th), number_of_cams=1)
    st.first_frame(0, 500)
    key = 0
    for i in range(1, 31):
        T = np.linalg.inv(steps[key]) @ steps[i]
        if st.tracked_frame(i, T[:3], int(inl[i]), 500):
            key = i
    assert st.result.keyframe_ids == want["keyframe_ids"] and 3 <= len(want["keyframe_ids"]) < 31
    assert np.allclose(np.array(st.result.poses_wrt_S), np.array(want["poses_wrt_S"]), atol=1e-12)
