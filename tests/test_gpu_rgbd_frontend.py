"""GPU, BASELINE config 5 batched: the RGB-D front-end (sos_frontend_create_rgbd / step_rgbd / submit_host_rgbd) at
640x480 and 2000 keypoints per frame, both depth encodings — store against sos_rgbd_backproject (bit-equal) and the
float64 oracle, temporal matches against cv2 BFMatcher + sort + gate, RANSAC against the oracle on the store's float32
points, the LM pose, agreement with the per-pair mirror (RGBDFrame + TrackerRGBDSE3), graph / eager / host paths over
consecutive steps, BatchedVO in keyframe mode against the sequential oracle loop, and the edge cases."""
import ctypes as C
import math

import cv2
import numpy as np
import pytest
import torch

from oracle import driver as odriver, geometry, rgbd as orgbd

pytestmark = pytest.mark.gpu

B = 8
MAX_KP = 2000
THR = 1.0 - math.cos(math.radians(5.0))
ENC = [pytest.param(True, id="Z"), pytest.param(False, id="radial")]


def seq_for(depth_is_Z, n_frames, seed=None):
    from vo_single_camera_sos_b200 import synth
    return synth.make_rgbd_sequence(n_frames, 2000, depth_is_Z, (0 if depth_is_Z else 2) if seed is None else seed)


def make_fe(ctx, seq, batch=B, solver=0, **kw):
    from vo_single_camera_sos_b200 import ops, pyopengv
    from vo_single_camera_sos_b200.frontend import Frontend, RgbdFrontendConfig
    hyp = pyopengv.hypothesis_list(210, 0, 4 if solver == ops.SOLVER_P3P else 3)
    kw.setdefault("refine_iters", 60)
    cfg = RgbdFrontendConfig(batch=batch, cam=seq.cam_vector(), max_kp=MAX_KP, solver=solver, **kw)
    return Frontend(ctx, cfg, None, torch.from_numpy(hyp.view(np.int32)).cuda()), hyp


def dev(inp):
    return [torch.from_numpy(np.ascontiguousarray(inp[k])).cuda() for k in ("depth", "px", "desc", "n_kp")]


def host(buf):
    return {k: (v.cpu().numpy() if isinstance(v, torch.Tensor) else v) for k, v in buf.items()}


def camd(seq):
    return dict(zip(geometry.RGBD_FIELDS, seq.cam_vector()))


def store_pts(buf, slot):
    """The store's float32 points of a slot as (xyz, bearing), for the oracle's pts= hook."""
    n = int(buf["n"][slot])
    return buf["xyz"][slot, :n], buf["b_top"][slot, :n]


def frame_oracle(seq, inp, b):
    n = int(inp["n_kp"][b])
    return orgbd.rgbd_frame(camd(seq), inp["depth"][b], inp["px"][b, :n], inp["desc"][b, :n])


def with_outside_keypoints(inp):
    """Frame 2: keypoints whose truncated pixel lies outside the map and a NaN coordinate (dropped), and two just inside."""
    inp["px"][2, :6] = [[-3.5, 10.0], [640.2, 5.0], [10.0, 480.0], [-0.5, -0.5], [np.nan, 3.0], [639.99, 479.99]]
    inp["depth"][2, 0, 0] = inp["depth"][2, 479, 639] = 2.5
    return inp


@pytest.mark.parametrize("depth_is_Z", ENC)
def test_store_equals_backproject_and_oracle(ctx, depth_is_Z):
    seq = seq_for(depth_is_Z, B)
    inp = with_outside_keypoints(seq.inputs(range(B), MAX_KP))
    fe, _ = make_fe(ctx, seq)
    d = dev(inp)
    fe.step_rgbd(*d)
    torch.cuda.synchronize()
    buf = host(fe.buffers())
    assert "pano" not in buf and "uv_bot" not in buf and "cam" not in buf and buf["uv_c"].shape[0] == 1
    for b in range(B):
        o = frame_oracle(seq, inp, b)
        s, n = b + 1, int(buf["n"][b + 1])
        assert n == len(o["src"]) > 1000 and buf["stats"][b, 0] == n
        assert np.array_equal(buf["src_top"][s, :n], o["src"])                     # valid set and order
        assert np.array_equal(buf["uv_top"][s, :n], inp["px"][b][o["src"]])
        assert np.array_equal(buf["desc_c"][0, s, :n].view(np.uint8).reshape(n, 32), inp["desc"][b][o["src"]])
        np.testing.assert_allclose(buf["xyz"][s, :n], o["xyz"], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(buf["b_top"][s, :n], o["b"], rtol=1e-4, atol=1e-6)
        # bit-equal to sos_rgbd_backproject on the same pixels
        px = inp["px"][b][o["src"]]
        u = torch.from_numpy(np.trunc(px[:, 0]).astype(np.int32)).cuda()
        v = torch.from_numpy(np.trunc(px[:, 1]).astype(np.int32)).cuda()
        xyz, bearing, valid = ctx.rgbd_backproject(seq.cam_vector(), d[0][b:b + 1], u, v, 0.8, 7.0)
        assert valid.cpu().numpy().all()
        assert np.array_equal(xyz.cpu().numpy().reshape(-1, 3), buf["xyz"][s, :n])
        assert np.array_equal(bearing.cpu().numpy().reshape(-1, 3), buf["b_top"][s, :n])
    kept = buf["src_top"][3, :buf["n"][3]]
    assert not np.isin([0, 1, 2, 4], kept).any() and np.isin([3, 5], kept).all()   # (-0.5, -0.5) truncates to (0, 0)
    fe.close()


@pytest.mark.parametrize("depth_is_Z", ENC)
def test_pairs_equal_oracle_and_mirror(ctx, depth_is_Z, monkeypatch):
    """Matches (pairs and order), RANSAC (best hypothesis, count, inlier mask) and the LM pose of every pair against the
    oracle on the store's float32 points, and against the per-pair mirror."""
    from omnistereo import pose_est_tools
    from omnistereo.camera_models import RGBDCamModel
    seq = seq_for(depth_is_Z, B)
    inp = seq.inputs(range(B), MAX_KP)
    fe, hyp = make_fe(ctx, seq)
    fe.step_rgbd(*dev(inp))
    torch.cuda.synchronize()
    buf = host(fe.buffers())
    cap = MAX_KP
    # pair 0 tracks frame 0 against the empty slot 0 (nothing carried yet): a tracking failure
    assert buf["n_corr"][0] == 0 and buf["best_hyp"][0] == -1 and buf["stats"][0, 1] == 0
    # the mirror on the same frames
    c = seq.cam
    cam = RGBDCamModel(fx=c["fx"], fy=c["fy"], center_x=c["center_x"], center_y=c["center_y"], depth_is_Z=depth_is_Z,
                       units="m")
    tracker = pose_est_tools.TrackerRGBDSE3(cam)
    assert tracker.max_horizontal_diff_f2f_matches == 319.5
    seen = {}
    real = pose_est_tools.absolute_pose_ransac

    def spy(*a, **k):
        seen["out"] = real(*a, **k)
        return seen["out"]
    monkeypatch.setattr(pose_est_tools, "absolute_pose_ransac", spy)
    rgb = np.zeros((480, 640, 3), np.uint8)
    mframes = []
    for b in range(B):
        n = int(inp["n_kp"][b])
        kp = [cv2.KeyPoint(float(x), float(y), 7.0) for x, y in inp["px"][b, :n]]
        mframes.append(pose_est_tools.RGBDFrame(cam, rgb, inp["depth"][b], b, features=(kp, inp["desc"][b, :n])))
    for i in range(1, B):
        ref, cur = frame_oracle(seq, inp, i - 1), frame_oracle(seq, inp, i)
        pts = {id(ref): store_pts(buf, i), id(cur): store_pts(buf, i + 1)}
        o = orgbd.rgbd_track_pair(ref, cur, hyp, THR, 319.5, pts=lambda f: pts[id(f)])
        nc = o["n_corr"]
        assert buf["n_corr"][i] == nc == buf["tm_pair_count"][i] and buf["stats"][i, 1] == nc
        q0 = int(buf["tm_q_start"][i])
        qi, ti = o["pairs"]
        assert np.array_equal(buf["tm_pair_q"][q0:q0 + nc] - (i + 1) * cap, qi)
        assert np.array_equal(buf["tm_pair_t"][q0:q0 + nc] - i * cap, ti)
        assert o["best_hyp"] >= 0 and buf["best_hyp"][i] == o["best_hyp"] and buf["best_count"][i] == o["best_count"]
        assert np.array_equal(buf["inlier_mask"][i, :nc].astype(bool), o["mask"])
        np.testing.assert_allclose(buf["pose"][i], o["refit"], rtol=0, atol=1e-6)
        # the mirror: same inliers and pose
        ok, msg = tracker.track_frame(mframes[i - 1], mframes[i])
        assert ok, msg
        assert tracker.num_tracked_correspondences == buf["best_count"][i]
        assert np.array_equal(seen["out"][1], np.flatnonzero(buf["inlier_mask"][i, :nc]))
        np.testing.assert_allclose(mframes[i].T_frame_wrt_tracking_ref_frame[:3], buf["pose"][i], rtol=0, atol=1e-6)
    fe.close()


def test_p3p_solver_equals_oracle(ctx):
    from vo_single_camera_sos_b200 import ops
    seq = seq_for(True, B)
    inp = seq.inputs(range(B), MAX_KP)
    fe, hyp = make_fe(ctx, seq, solver=ops.SOLVER_P3P, refit=ops.REFINE_NONE)
    fe.step_rgbd(*dev(inp))
    torch.cuda.synchronize()
    buf = host(fe.buffers())
    for i in (1, 4, 7):
        ref, cur = frame_oracle(seq, inp, i - 1), frame_oracle(seq, inp, i)
        pts = {id(ref): store_pts(buf, i), id(cur): store_pts(buf, i + 1)}
        o = orgbd.rgbd_track_pair(ref, cur, hyp, THR, 319.5, solver="p3p", refine="none", pts=lambda f: pts[id(f)])
        nc = o["n_corr"]
        assert o["best_hyp"] >= 0 and buf["best_hyp"][i] == o["best_hyp"] and buf["best_count"][i] == o["best_count"]
        assert np.array_equal(buf["inlier_mask"][i, :nc].astype(bool), o["mask"])
        assert np.array_equal(buf["pose"][i], buf["ransac_pose"][i])
        np.testing.assert_allclose(buf["pose"][i], o["pose"], rtol=0, atol=1e-4)
    fe.close()


@pytest.mark.parametrize("depth_is_Z", ENC)
def test_graph_eager_and_host_paths_bit_equal(ctx, depth_is_Z):
    """Three consecutive steps (the last frame of a step is the reference of the next one's first pair)."""
    seq = seq_for(depth_is_Z, 3 * B)
    batches = [seq.inputs(range(k * B, (k + 1) * B), MAX_KP) for k in range(3)]
    fg, _ = make_fe(ctx, seq)
    fx, _ = make_fe(ctx, seq)
    fx.set_graph(False)
    fh, _ = make_fe(ctx, seq)
    d_in = dev(batches[0])           # fixed device inputs: from the second step on, the graph step replays its graph
    keys = ("pose", "ransac_pose", "stats", "best_hyp", "best_count", "n_corr", "n", "tm_pair_count", "refine_stats")
    pinned = [{k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in bt.items()} for bt in batches]
    for k, bt in enumerate(batches):
        for t, a in zip(d_in, dev(bt)):
            t.copy_(a)
        fg.step_rgbd(*d_in)
        fx.step_rgbd(*d_in)
        p = pinned[k]
        poses, stats = fh.step_host_rgbd(p["depth"], p["px"], p["desc"], p["n_kp"])
        torch.cuda.synchronize()
        g, x, h = host(fg.buffers()), host(fx.buffers()), host(fh.buffers())
        for name in keys:
            assert np.array_equal(g[name], x[name], equal_nan=True), (k, name)
            assert np.array_equal(g[name], h[name], equal_nan=True), (k, name)
        assert np.array_equal(poses, g["pose"], equal_nan=True) and np.array_equal(stats, g["stats"])
        for s in range(B + 1):
            n = int(g["n"][s])
            for name in ("xyz", "b_top", "uv_top", "src_top"):
                assert np.array_equal(g[name][s, :n], h[name][s, :n], equal_nan=True), (k, name, s)
                assert np.array_equal(g[name][s, :n], x[name][s, :n], equal_nan=True), (k, name, s)
        for i in range(B):
            nc = int(g["n_corr"][i])
            assert np.array_equal(g["inlier_mask"][i, :nc], h["inlier_mask"][i, :nc])
        if k > 0:   # the carried frame: pair 0 tracks against the previous step's last frame
            assert g["n_corr"][0] > 100 and g["best_hyp"][0] >= 0
    assert fg.buffers()["launches_per_step"] > 0
    h2d, d2h = fh.host_bytes()
    assert h2d == B * (480 * 640 * 4 + MAX_KP * 40 + 4) and d2h == B * 64
    for f in (fg, fx, fh):
        f.close()


@pytest.mark.parametrize("depth_is_Z", ENC)
def test_batched_vo_keyframes_equal_sequential_oracle(ctx, depth_is_Z):
    from vo_single_camera_sos_b200.driver import BatchedVO, KeyframePolicy
    from vo_single_camera_sos_b200.frontend import RgbdFrontendConfig
    from vo_single_camera_sos_b200 import pyopengv
    n_frames = 40
    seq = seq_for(depth_is_Z, n_frames)
    hyp = pyopengv.hypothesis_list(210, 0)
    th = dict(odriver.INDOOR, pos_min=0.06)
    want = orgbd.run_vo(seq.frames, camd(seq), hyp, THR, 319.5, thresholds=th, refine="lm")
    assert want["status"] == "ok" and 5 <= len(want["keyframe_ids"]) < n_frames
    for dist, ang, *_ in want["decisions"]:   # no decision within 100x the pose tolerance of a threshold
        assert abs(dist - th["pos_min"]) > 1e-4 and abs(dist - th["pos_max"]) > 1e-4 and abs(ang - th["ang_max"]) > 1e-4
    cfg = RgbdFrontendConfig(batch=B, cam=seq.cam_vector(), max_kp=MAX_KP, keyframe_mode=True, refine_iters=60)
    vo = BatchedVO(ctx, cfg, None, torch.from_numpy(hyp.view(np.int32)).cuda(), KeyframePolicy(**th))
    assert vo.number_of_cams == 1 and vo.min_correspondences == 6
    frames = [dict(depth=f["depth"], px=np.pad(f["px"], ((0, MAX_KP - len(f["px"])), (0, 0))),
                   desc=np.pad(f["desc"], ((0, MAX_KP - len(f["desc"])), (0, 0))), n_kp=len(f["px"])) for f in seq.frames]
    res = vo.run(frames)
    assert res.status == "ok"
    assert res.keyframe_ids == want["keyframe_ids"]
    assert res.tracked == want["tracked"]
    assert np.allclose(np.array(res.poses_wrt_S), np.array(want["poses_wrt_S"]), atol=1e-4)
    vo.close()


def test_edge_cases(ctx):
    from vo_single_camera_sos_b200 import ops, workload
    from vo_single_camera_sos_b200._lib import SosError
    from vo_single_camera_sos_b200.driver import BatchedVO, KeyframePolicy
    from vo_single_camera_sos_b200.frontend import RgbdFrontendConfig
    from vo_single_camera_sos_b200 import pyopengv
    seq = seq_for(True, B)
    inp = seq.inputs(range(B), MAX_KP)
    inp["n_kp"][3] = 0                  # a frame with no keypoints
    inp["depth"][5] = 0.0               # an all-zero depth map: no valid keypoint
    fe, _ = make_fe(ctx, seq)
    fe.step_rgbd(*dev(inp))
    torch.cuda.synchronize()
    buf = host(fe.buffers())
    assert buf["n"][4] == 0 and buf["n"][6] == 0 and buf["n"][3] > 1000
    for i in (3, 4, 5, 6):              # pairs touching an empty frame have no correspondences and no model
        assert buf["n_corr"][i] == 0 and buf["best_hyp"][i] == -1 and buf["best_count"][i] <= 0
    assert buf["best_hyp"][2] >= 0 and buf["best_hyp"][7] >= 0
    # n_kp above max_kp: refused on the host path, clamped on the device path
    bad = {k: v.copy() for k, v in inp.items()}
    bad["n_kp"][1] = MAX_KP + 1
    with pytest.raises(ValueError):
        fe.step_host_rgbd(bad["depth"], bad["px"], bad["desc"], bad["n_kp"])
    lib = ctx.lib
    t = C.c_int()
    ptr = lambda a: a.ctypes.data
    assert lib.sos_frontend_submit_host_rgbd(fe._h, ptr(bad["depth"]), ptr(bad["px"]), ptr(bad["desc"]), ptr(bad["n_kp"]),
                                             C.byref(t)) == -1
    fe.reset()
    clamp = {k: v.copy() for k, v in inp.items()}
    clamp["n_kp"][1] = MAX_KP + 7
    fe.step_rgbd(*dev(clamp))
    torch.cuda.synchronize()
    assert fe.buffers()["n"][2].item() == buf["n"][2]
    fe.close()
    # fewer than 6 correspondences: tracking failure in the driver
    frames = []
    for b in range(B):
        n = 5 if b == 4 else MAX_KP
        frames.append(dict(depth=inp["depth"][b] if b != 5 else seq.frames[5]["depth"], px=inp["px"][b].copy(),
                           desc=inp["desc"][b].copy(), n_kp=n))
    hyp = pyopengv.hypothesis_list(210, 0)
    cfg = RgbdFrontendConfig(batch=4, cam=seq.cam_vector(), max_kp=MAX_KP, keyframe_mode=True)
    vo = BatchedVO(ctx, cfg, None, torch.from_numpy(hyp.view(np.int32)).cuda(), KeyframePolicy(pos_min=0.06))
    res = vo.run(frames)
    assert res.status.startswith("tracking failed at frame 4") and res.frame_ids == [0, 1, 2, 3]
    vo.close()
    # SOS and RGB-D calls refuse each other's front-end (SOS_ERR_INVALID = -1 in C, TypeError in Python)
    rg, _ = make_fe(ctx, seq, batch=2)
    w = workload.build(ctx, "tiny", batch=2, n_frames=2, seed=1, score_mode=ops.SCORE_BEARING)
    sf = w.frontend(ctx)
    z = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    p = z.data_ptr()
    assert lib.sos_frontend_step(rg._h, p, p, p, p, p, p, p) == -1
    assert lib.sos_frontend_submit_host(rg._h, p, p, p, p, p, p, p, C.byref(t)) == -1
    assert lib.sos_frontend_step_host(rg._h, p, p, p, p, p, p, p, p, p) == -1
    assert lib.sos_frontend_set_detector(rg._h, p, p, p) == -1
    assert lib.sos_frontend_step_images(rg._h, p) == -1
    assert lib.sos_frontend_submit_host_images(rg._h, p, C.byref(t)) == -1
    assert lib.sos_frontend_get_features(rg._h, p) == -1
    assert lib.sos_frontend_step_rgbd(sf._h, p, p, p, p) == -1
    assert lib.sos_frontend_submit_host_rgbd(sf._h, p, p, p, p, C.byref(t)) == -1
    with pytest.raises(TypeError):
        rg.step_images(z)
    with pytest.raises(TypeError):
        sf.step_rgbd(z, z, z, z)
    # the calls both kinds share
    rg.set_graph(True)
    rg.reset()
    rg.profile_begin()
    rg.step_rgbd(*dev(seq.inputs(range(2), MAX_KP)))
    prof = rg.profile_end()
    assert [n for n, _ in prof][0] == "rgbd_store_kernel" and all(ms >= 0 for _, ms in prof)
    with pytest.raises(SosError):
        rg.set_ref_slots([0, 0])        # keyframe mode only
    rg.close()
    sf.close()
