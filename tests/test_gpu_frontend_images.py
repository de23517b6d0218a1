"""GPU: images-in steps of the batched front-end (sos_frontend_set_detector / step_images / submit_host_images).
The features detected inside the step equal features.FeatureFront.detect on the step's own panoramas bit for bit, and
everything after them equals a second front-end stepped by sos_frontend_step on those features."""
import ctypes as C
import time

import cv2
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STORE_AND_RANSAC = ("pano", "st_pair_count", "st_pair_q", "st_pair_t", "uv_c", "b_top", "b_bot", "xyz", "src_top", "src_bot",
                    "n", "desc_c", "tm_pair_count", "tm_pair_q", "tm_pair_t", "p_ref", "p_cur", "f_cur", "cam", "n_corr",
                    "n_corr_top", "ransac_pose", "pose", "best_hyp", "best_count", "n_refit", "inlier_mask", "stats",
                    "overflow")


def masks_for(w, overlap: int):
    """Azimuthal masks of both views restricted to the eroded valid panorama (as scripts/bench_images.py builds them);
    overlap > 0 widens every bucket by that many columns on each side, so that neighbouring masks share pixels."""
    from vo_single_camera_sos_b200.features import azimuthal_masks
    rows, cols, nb = w.cfg.pano_rows, w.cfg.pano_cols, w.cfg.n_buckets
    valid = ((w.lut >> 48) & 0xF) != 0
    out = []
    for view in range(2):
        v = cv2.erode(valid[view].cpu().numpy().astype(np.uint8), np.ones((7, 7), np.uint8)).astype(bool)
        m = azimuthal_masks(rows, cols, nb)
        if overlap:
            k = np.ones((1, 2 * overlap + 1), np.uint8)
            m = np.stack([cv2.dilate(mk, k, borderType=cv2.BORDER_CONSTANT, borderValue=0) for mk in m])
        out.append(m & (v[None] * 255).astype(np.uint8))
    return out


def corners_per_bucket(w):
    from vo_single_camera_sos_b200 import workload
    return min(w.cfg.max_feat_per_bucket, workload.CONFIGS[w.name]["feat"] // 12 + 1)


def render(ctx, w, first, count):
    from vo_single_camera_sos_b200 import workload
    r = workload.DeviceRenderer(ctx, w)
    return torch.stack([r.render(w.trajectory[first + i]) for i in range(count)]).contiguous()


def feature_front(ctx, w, masks, N, median):
    from vo_single_camera_sos_b200.features import FeatureFront
    return FeatureFront(ctx, masks[0], masks[1], corners_per_bucket=N, max_feat_per_view=w.cfg.max_feat_per_view,
                        median=median)


def feats_tuple(f):
    return tuple(f[k].clone() for k in ("px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot"))


def assert_same(a: torch.Tensor, b: torch.Tensor, what):
    assert a.shape == b.shape, what
    assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes(), what


@pytest.mark.parametrize("name,overlap,median,B,F", [("tiny", 0, True, 3, None), ("tiny", 3, False, 3, None),
                                                     ("tiny", 0, True, 3, 40), ("c1", 0, True, 2, None),
                                                     ("c1", 4, False, 2, None), ("c2", 0, True, 2, None),
                                                     ("c2", 6, False, 1, None)])
def test_features_equal_feature_front(ctx, name, overlap, median, B, F):
    """F: max_feat_per_view small enough that the clamp drops rows (None: the workload's own, which keeps them all)."""
    import dataclasses
    from vo_single_camera_sos_b200 import ops, workload
    w = workload.build(ctx, name, batch=B, n_frames=2 * B + 1, seed=11, score_mode=ops.SCORE_BEARING)
    if F is not None:
        w.cfg = dataclasses.replace(w.cfg, max_feat_per_view=F)
    masks = masks_for(w, overlap)
    if overlap:
        assert (np.count_nonzero(masks[0], axis=0) > 1).any()
    N = corners_per_bucket(w)
    fe = w.frontend(ctx)
    fe.set_detector(masks[0], masks[1], N, median=median)
    front = feature_front(ctx, w, masks, N, median)
    for step in range(2):
        fe.step_images(render(ctx, w, step * B, B))
        torch.cuda.synchronize()
        want = front.detect(fe.buffers()["pano"].clone())
        f = fe.features()
        for key, ref in zip(("px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot"), want):
            assert_same(f[key], ref, (step, key))
        st = f["detect_stats"].cpu().numpy()
        boff = np.stack([f["boff_top"].cpu().numpy(), f["boff_bot"].cpu().numpy()], 1)   # [B, 2, nb+1]
        Fv = w.cfg.max_feat_per_view
        assert (st[..., 3] == 0).all() and (st[..., 1] <= st[..., 0]).all()
        assert np.array_equal(boff[..., -1], np.minimum(st[..., 1], Fv))
        assert np.array_equal(st[..., 2], np.maximum(st[..., 1] - Fv, 0))
        assert (boff[..., -1] > 0).all()
        assert (st[..., 2] > 0).any() if F is not None else (st[..., 2] == 0).all()
    fe.close()


@pytest.mark.parametrize("keyframe,graph", [(False, True), (False, False), (True, True)])
def test_rest_of_step_equals_feature_step(ctx, keyframe, graph):
    """Every buffer after step_images equals a front-end of the same configuration stepped by sos_frontend_step on the
    detected features, over alternating omni buffers (graph replay and eager); keyframe mode with promote + retrack."""
    from vo_single_camera_sos_b200 import ops, workload
    B = 3
    w = workload.build(ctx, "tiny", batch=B, n_frames=3 * B + 1, seed=4, score_mode=ops.SCORE_BEARING)
    w.cfg.keyframe_mode = keyframe
    masks = masks_for(w, 0)
    fe, ref = w.frontend(ctx), w.frontend(ctx)
    fe.set_graph(graph)
    ref.set_graph(graph)
    fe.set_detector(masks[0], masks[1], corners_per_bucket(w))
    omnis = [render(ctx, w, s * B, B) for s in range(2)]
    for step in range(4):
        omni = omnis[step % 2]
        fe.step_images(omni)
        feats = feats_tuple(fe.features())
        ref.step(omni, *feats)
        if keyframe and step == 1:
            for h in (fe, ref):
                h.promote(2)
                h.set_ref_slots([0, -1, 0])
                h.retrack()
        torch.cuda.synchronize()
        a, b = fe.buffers(), ref.buffers()
        for k in STORE_AND_RANSAC:
            assert_same(a[k], b[k], (step, k))
    # the graph cache tells an images-in step from a feature step on the same omni and on the front-end's own features
    f = fe.features()
    fe.step(omnis[0], *(f[k] for k in ("px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot")))
    ref.step(omnis[0], *feats_tuple(f))
    torch.cuda.synchronize()
    a, b = fe.buffers(), ref.buffers()
    for k in STORE_AND_RANSAC:
        assert_same(a[k], b[k], ("feature step", k))
    fe.close(); ref.close()


def test_detector_does_not_invalidate_captured_feature_steps(ctx):
    """A feature step captured before the detector is attached replays correctly after images-in steps on large panoramas
    with small feature capacities (detection scratch far larger than what the feature steps use): the same sequence on a
    front-end that never had a detector gives the same buffers."""
    import dataclasses
    from vo_single_camera_sos_b200 import frontend, ops, workload
    B = 2
    w = workload.build(ctx, "c1", batch=B, n_frames=2 * B + 1, seed=12, score_mode=ops.SCORE_BEARING)
    cfg = dataclasses.replace(w.cfg, cap=64, max_feat_per_view=256, max_feat_per_bucket=32)
    masks = masks_for(w, 0)
    make = lambda: frontend.Frontend(ctx, cfg, w.lut, w.hyp)
    fe, ref, src = make(), make(), make()
    src.set_detector(masks[0], masks[1], 16)
    omni_a, omni_b = render(ctx, w, 0, B), render(ctx, w, B, B)
    src.step_images(omni_a)
    feats_a = feats_tuple(src.features())
    for h in (fe, ref):
        h.step(omni_a, *feats_a)                     # eager run + capture
        h.step(omni_a, *feats_a)                     # replay
    fe.set_detector(masks[0], masks[1], 16)
    fe.step_images(omni_b)
    feats_b = feats_tuple(fe.features())
    ref.step(omni_b, *feats_b)
    for h in (fe, ref):
        h.step(omni_a, *feats_a)                     # the graph captured before the detector, if still valid
    torch.cuda.synchronize()
    a, b = fe.buffers(), ref.buffers()
    for k in STORE_AND_RANSAC:
        assert_same(a[k], b[k], k)
    fe.close(); ref.close(); src.close()


@pytest.mark.parametrize("upload", ["bands", "full"])
def test_host_images_equals_device_images(ctx, upload, monkeypatch):
    from vo_single_camera_sos_b200 import workload
    if upload == "full":
        monkeypatch.setenv("SOS_FULL_UPLOAD", "1")
    else:
        monkeypatch.delenv("SOS_FULL_UPLOAD", raising=False)
    B = 2
    w = workload.build(ctx, "tiny", batch=B, n_frames=3 * B + 1, seed=6)
    masks = masks_for(w, 0)
    N = corners_per_bucket(w)
    fe_dev, fe_host = w.frontend(ctx), w.frontend(ctx)
    for h in (fe_dev, fe_host):
        h.set_detector(masks[0], masks[1], N)
    omnis = [render(ctx, w, s * B, B) for s in range(3)]
    want = []
    for o in omnis:
        fe_dev.step_images(o)
        torch.cuda.synchronize()
        b = fe_dev.buffers()
        want.append((b["pose"].cpu().numpy().copy(), b["stats"].cpu().numpy().copy()))
    pinned = [o.cpu().pin_memory() for o in omnis]
    t0 = fe_host.submit_host_images(pinned[0])
    t1 = fe_host.submit_host_images(pinned[1])
    got = [fe_host.wait_host(t0), fe_host.wait_host(t1), fe_host.step_host_images(pinned[2])]
    for (p, s), (wp, ws) in zip(got, want):
        assert np.array_equal(s, ws)
        assert np.array_equal(p, wp, equal_nan=True)
    full = B * w.cfg.src_h * w.cfg.src_w * 3
    nbytes = fe_host.host_images_bytes()
    assert nbytes == full if upload == "full" else 0 < nbytes <= full
    fe_dev.close(); fe_host.close()


def test_candidate_overflow_drops_only_that_mask(ctx):
    """Frame 0 is noise (more than 16 384 candidates under mask 0 of the top view), frame 1 smooth texture: the step
    succeeds, frame 0 gets no corners from mask 0 and detect_stats counts the refused mask, frame 1 equals FeatureFront
    on frame 1 alone."""
    from oracle import gft as ogft
    from vo_single_camera_sos_b200 import ops, workload
    B = 2
    w = workload.build(ctx, "c1", batch=B, n_frames=B + 1, seed=8, score_mode=ops.SCORE_BEARING)
    rows, cols, nb = w.cfg.pano_rows, w.cfg.pano_cols, w.cfg.n_buckets
    valid = ((w.lut >> 48) & 0xF).cpu().numpy() != 0
    masks = []
    for view in range(2):
        # one mask over the panorama, away from ORB's 31-pixel border, the others empty
        v = cv2.erode(valid[view].astype(np.uint8), np.ones((7, 7), np.uint8)).astype(bool)
        v[:40] = v[-40:] = False
        m = np.zeros((nb, rows, cols), np.uint8)
        m[0][v] = 255
        masks.append(m)
    N = 100
    fe = w.frontend(ctx)
    fe.set_detector(masks[0], masks[1], N, median=False)
    rng = np.random.default_rng(3)
    shape = (w.cfg.src_h, w.cfg.src_w, 3)
    smooth = cv2.GaussianBlur(rng.integers(0, 256, shape, dtype=np.uint8), (0, 0), 6.0)
    omni = torch.from_numpy(np.stack([rng.integers(0, 256, shape, dtype=np.uint8), smooth])).to(ctx.device)
    fe.step_images(omni)
    torch.cuda.synchronize()
    pano = fe.buffers()["pano"].clone()
    over = []
    for view in range(2):
        n0, n1 = (len(ogft.candidates(ogft.corner_min_eigenval(cv2.cvtColor(pano[b, view].cpu().numpy(), cv2.COLOR_BGR2GRAY)),
                                      masks[view][0], 0.01)) for b in range(2))
        assert n1 < 16384
        over.append(n0 > 16384)
    assert over[0]                                   # the top view of frame 0 at least
    f = fe.features()
    st = f["detect_stats"].cpu().numpy()
    assert np.array_equal(st[0, :, 3], np.array(over, np.int32)) and (st[1, :, 3] == 0).all()
    assert (st[0, over, 0] == 0).all()
    for key, view in (("boff_top", 0), ("boff_bot", 1)):
        if over[view]:
            assert (f[key][0].cpu().numpy() == 0).all()
    front = feature_front(ctx, w, masks, N, False)
    want = front.detect(pano[1:2].contiguous())
    for key, ref in zip(("px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot"), want):
        assert_same(f[key][1:2], ref, key)
    assert int(f["boff_top"][1, -1]) > 0
    fe.close()


def test_step_images_does_not_wait_for_the_device(ctx):
    from vo_single_camera_sos_b200 import workload
    B = 2
    w = workload.build(ctx, "tiny", batch=B, n_frames=B + 1, seed=2)
    masks = masks_for(w, 0)
    fe = w.frontend(ctx)
    fe.set_detector(masks[0], masks[1], corners_per_bucket(w))
    omni = render(ctx, w, 0, B)
    for _ in range(2):
        fe.step_images(omni)                         # the first call runs eagerly, sizes the arena and captures
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    torch.cuda._sleep(int(4e8))                      # about 200 ms of the GPU clock on the caller's stream
    fe.step_images(omni)
    t_call = time.perf_counter() - t0
    torch.cuda.synchronize()
    t_all = time.perf_counter() - t0
    assert t_all > 0.1 and t_call < 0.25 * t_all, (t_call, t_all)
    fe.close()


def test_argument_refusals(ctx):
    import dataclasses
    from vo_single_camera_sos_b200 import frontend, workload
    from vo_single_camera_sos_b200._lib import SosError, check
    w = workload.build(ctx, "tiny", batch=2, n_frames=3, seed=1)
    masks = masks_for(w, 0)
    fe = w.frontend(ctx)
    with pytest.raises(SosError) as e:
        fe.step_images(render(ctx, w, 0, 2))         # no detector yet
    assert e.value.code == -1
    with pytest.raises(SosError):
        fe.features()
    with pytest.raises(SosError):
        fe.set_detector(masks[0], masks[1], w.cfg.max_feat_per_bucket + 1)
    d = frontend._DetectConfig(10, 1, 0.01, 5.0)
    with pytest.raises(SosError):
        check(ctx.lib.sos_frontend_set_detector(fe._h, C.byref(d), None, None))
    fe.close()
    # a front-end of 1-channel images, and one with 33 buckets
    for field, value in (("channels", 1), ("n_buckets", 33)):
        cfg = dataclasses.replace(w.cfg, **{field: value})
        h = frontend.Frontend(ctx, cfg, w.lut, w.hyp)
        m = torch.zeros((cfg.n_buckets, cfg.pano_rows, cfg.pano_cols), dtype=torch.uint8, device=ctx.device)
        with pytest.raises(SosError) as e:
            h.set_detector(m, m, 10)
        assert e.value.code == -4, field
        h.close()
