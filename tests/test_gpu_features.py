"""GPU: the image-in front-end (SURVEY §8f N3 chained in front of the hot path): feature arrays produced on the device
from rendered omni images equal what the reference's OpenCV calls give on the same panoramas (the corner lists exactly
those of oracle/gft.py on cv2's median and gray), and the poses that come out
of Frontend.step on them follow the ground-truth motion."""
import cv2
import numpy as np
import pytest
import torch

from oracle import gft as ogft

pytestmark = pytest.mark.gpu


def test_image_in_front_end(ctx):
    from vo_single_camera_sos_b200 import ops, workload
    from vo_single_camera_sos_b200.features import FeatureFront, azimuthal_masks, step_images
    B, N = 2, 120
    w = workload.build(ctx, "c1", batch=B, n_frames=2 * B + 1, seed=2, score_mode=ops.SCORE_BEARING)
    w.cfg.n_hyp = w.cfg.n_hyp
    rows, cols = w.cfg.pano_rows, w.cfg.pano_cols
    valid = ((w.lut >> 48) & 0xF) != 0                                  # [2, rows, cols]: panorama pixels with a source
    masks = []
    for view in range(2):
        v = valid[view].cpu().numpy()
        v = cv2.erode(v.astype(np.uint8), np.ones((7, 7), np.uint8)).astype(bool)
        masks.append(azimuthal_masks(rows, cols, 12) & (v[None] * 255).astype(np.uint8))
    front = FeatureFront(ctx, masks[0], masks[1], corners_per_bucket=N, max_feat_per_view=w.cfg.max_feat_per_view)
    assert N <= w.cfg.max_feat_per_bucket
    renderer = workload.DeviceRenderer(ctx, w)
    fe = w.frontend(ctx)
    poses = []
    for step in range(2):
        omni = torch.stack([renderer.render(w.trajectory[step * B + i]) for i in range(B)]).contiguous()
        feats = step_images(fe, front, omni, w.lut)
        torch.cuda.synchronize()
        buf = fe.buffers()
        poses.append((buf["pose"].cpu().numpy().copy(), buf["stats"].cpu().numpy().copy()))
        if step == 0:
            # ---- the feature arrays against the reference's call sequence on the same panorama (frame 0, both views)
            pano = buf["pano"].cpu().numpy()
            for view, (px, ds, boff) in enumerate((feats[0:3], feats[3:6])):
                px, ds, boff = px.cpu().numpy(), ds.cpu().numpy(), boff.cpu().numpy()
                gray = cv2.cvtColor(cv2.medianBlur(pano[0, view], 11), cv2.COLOR_BGR2GRAY)
                orb = cv2.ORB_create(nfeatures=N)
                eig = ogft.corner_min_eigenval(gray)
                total = same = 0
                for k in range(12):
                    # exactly: cv2 median and gray, then the oracle's Shi-Tomasi, then ORB.compute
                    want, _ = ogft.good_features(eig, masks[view][k], N, 0.01, 5.0)
                    got_px, got_ds = px[0, boff[0, k]:boff[0, k + 1]], ds[0, boff[0, k]:boff[0, k + 1]]
                    ko, do = orb.compute(gray, list(cv2.KeyPoint_convert(want))) if len(want) else ([], np.zeros((0, 32), np.uint8))
                    assert np.array_equal(got_px, np.array([kp.pt for kp in ko], np.float32).reshape(-1, 2)), (view, k)
                    assert np.array_equal(got_ds, do), (view, k)
                    # against cv2's own corner lists (its SIMD tail columns may decide a near-tie differently)
                    pts = cv2.goodFeaturesToTrack(image=gray, maxCorners=N, qualityLevel=0.01, minDistance=5, mask=masks[view][k],
                                                  useHarrisDetector=False)
                    if pts is None:
                        assert boff[0, k + 1] == boff[0, k]
                        continue
                    kr, dr = orb.compute(gray, list(cv2.KeyPoint_convert(pts.reshape(-1, 2))))
                    got_px, got_ds = px[0, boff[0, k]:boff[0, k + 1]], ds[0, boff[0, k]:boff[0, k + 1]]
                    assert abs(len(got_px) - len(kr)) <= 2
                    for a, b, da, db in zip(got_px, kr, got_ds, dr):
                        total += 1
                        if tuple(a) == b.pt:
                            same += 1
                            assert np.array_equal(da, db)
                assert total > 300 and same >= 0.97 * total, (view, same, total)
    # ---- poses of the second step follow the ground-truth motion (frame k wrt frame k - 1)
    pose, stats = poses[1]
    for i in range(B):
        k = B + i
        T_rel = np.linalg.inv(w.trajectory[k - 1]) @ w.trajectory[k]
        assert stats[i, 0] > 100 and stats[i, 2] > 50, stats[i]          # stereo correspondences, RANSAC inliers
        assert np.allclose(pose[i][:, :3], T_rel[:3, :3], atol=0.03), (i, pose[i], T_rel)
        assert np.allclose(pose[i][:, 3], T_rel[:3, 3], atol=0.05), (i, pose[i][:, 3], T_rel[:3, 3])
    fe.close()
