"""Golden vectors for the VO LOOP from the reference's own `run_VO` (pose_est_tools.py:1264-1678), run UNMODIFIED in the build
container on a rendered synthetic sequence:

    python -m oracle.gen_vo_golden          ->  tests/golden/vo_sequence.npz

What is the reference's and what is harness here:
  * reference (imported from /root/reference, not edited): the model classes built through their constructors, per-frame
    masking + remap, GFT + ORB feature detection, bucketed stereo matching, lifting, triangulation, range gate, temporal
    matching, the stacking of correspondences, the keyframe decision tree, pose chaining and the TUM / keyframe-id writers.
  * harness: the shims of oracle/_ref_shims.py, a `matplotlib.pyplot.get_cmap` stub, the `cv2.KeyPoint_convert` reshape shim
    (OpenCV 4.13 rejects the (N,1,2) array goodFeaturesToTrack returns, camera_models.py:1752), and — because OpenGV is not
    available — a `pyopengv` stub backed by oracle/p3p.py (RANSAC over the shared seeded hypothesis list with the reference's
    own argument list: bearings of the current frame, 3D points of the reference frame, rig) and oracle/ransac.py
    (Levenberg-Marquardt refinement).  RANSAC / refinement parity with OpenGV itself stays UNPINNED; what this golden pins is
    everything AROUND those two calls, driven end to end by the reference's loop.

The features the reference detected are recorded (detection is upstream of the hot path) so that oracle/driver.py and the
GPU driver can be fed exactly what the reference's loop saw.  TEST INFRASTRUCTURE ONLY.
"""
from __future__ import annotations

import contextlib
import io
import os
import shutil
import sys
import tempfile
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")

# nine frames keep vo_sequence.npz under 1 MB (the ORB descriptors, ~100 KB a frame, barely compress); the loop is causal, so
# these are the first nine frames of a longer run of the same sequence
N_FRAMES, WIDTH, HEIGHT, PANO_COLS, SEED, N_LANDMARKS = 9, 640, 480, 800, 3, 500
RANSAC_SEED = 0
ROOM_SCALE = 0.4
RANSAC_CALLS = []


def install_extra_shims():
    import cv2
    from . import _ref_shims, p3p, ransac
    _ref_shims.install()
    # matplotlib is not installed: run_VO imports get_cmap for point colours it never uses without a visualiser (:1394)
    if "matplotlib" not in sys.modules:
        mpl, plt = types.ModuleType("matplotlib"), types.ModuleType("matplotlib.pyplot")
        plt.get_cmap = lambda name: (lambda x: (0.0, 0.0, 0.0, 1.0))
        mpl.pyplot = plt
        sys.modules["matplotlib"], sys.modules["matplotlib.pyplot"] = mpl, plt
    # draw_matches_between_frames must return an image: track_frame writes it with cv2.imwrite (:818-819)
    sys.modules["omnistereo.common_plot"].draw_matches_between_frames = lambda *a, **k: np.zeros((2, 2, 3), np.uint8)
    # OpenCV 4.13: KeyPoint_convert wants (N, 2)
    if not getattr(cv2.KeyPoint_convert, "_sos_shim", False):
        orig = cv2.KeyPoint_convert

        def convert(arg, *a, **k):
            if isinstance(arg, np.ndarray) and arg.ndim == 3 and arg.shape[1] == 1:
                arg = arg.reshape(arg.shape[0], arg.shape[2])
            return orig(arg, *a, **k)
        convert._sos_shim = True
        cv2.KeyPoint_convert = convert

    # --- pyopengv stub backed by the oracle ------------------------------------------------------------------------
    m = sys.modules["pyopengv"]

    def hypothesis_list(n_hyp, seed=RANSAC_SEED, k=4):
        return np.random.default_rng(seed).integers(0, 2 ** 32, (int(n_hyp), k), dtype=np.uint64).astype(np.uint32)

    def rig_of(offsets, rotations):
        off = np.asarray(offsets, np.float64).reshape(-1, 3)
        rot = np.asarray(rotations, np.float64).reshape(-1, 3, 3)
        return np.concatenate([rot, off[:, :, None]], axis=2)

    def absolute_pose_noncentral_ransac(b, cam_idx, p, offsets, rotations, thr, iters):
        rig = rig_of(offsets, rotations)
        cam = np.asarray(cam_idx).reshape(-1).astype(np.uint8)
        M, h, c, inl, _ = p3p.ransac_p3p(np.asarray(p, np.float32)[:, :3], np.asarray(b, np.float32)[:, :3], cam, rig,
                                         hypothesis_list(iters), float(thr))
        # what the reference's tracker handed to "OpenGV" for this frame, and what came back (recorded for the tests)
        RANSAC_CALLS.append(dict(points=np.asarray(p, np.float64)[:, :3].copy(), bearings=np.asarray(b, np.float64)[:, :3].copy(),
                                 cam=cam.copy(), best_hyp=int(h), inliers=np.nonzero(inl)[0].astype(np.int64),
                                 pose=np.asarray(M, np.float64).copy()))
        return np.asarray(M, np.float64), np.nonzero(inl)[0].astype(np.int64)

    def absolute_pose_noncentral_optimize_nonlinear(b, cam_idx, p, offsets, rotations, t, R):
        rig = rig_of(offsets, rotations)
        cam = np.asarray(cam_idx).reshape(-1).astype(np.uint8)
        pose0 = np.hstack([np.asarray(R, np.float64).reshape(3, 3), np.asarray(t, np.float64).reshape(3, 1)])
        return ransac.refine_pose_lm(np.asarray(p, np.float32)[:, :3], np.asarray(b, np.float32)[:, :3],
                                     pose0.astype(np.float32), cam, rig)[0]

    m.absolute_pose_noncentral_ransac = absolute_pose_noncentral_ransac
    m.absolute_pose_noncentral_optimize_nonlinear = absolute_pose_noncentral_optimize_nonlinear


def reference_gums(rig, pano_cols, first_image):
    """A GUMStereo through the REFERENCE's constructors (SURVEY 8c recipe) with the synthetic rig's parameters."""
    from omnistereo.gum import GUM, GUMStereo
    models = []
    for g, z_axis, F in ((rig.gum_top, 1.0, rig.f_top), (rig.gum_bot, -1.0, rig.f_bot)):
        m = GUM(precalib_filename="/nonexistent", new_method=True, z_axis=z_axis, image_size_pixels=(rig.width, rig.height),
                center_uv_point=np.array([g["u_center"], g["v_center"]]))
        m.precalib_params.set_gum_params(xi1=g["xi1"], xi2=g["xi2"], xi3=g["xi3"])
        m.precalib_params.set_generalized_cam_params(gamma1=g["gamma1"], gamma2=g["gamma2"], alpha_c=g["alpha_c"],
                                                     u_center=g["u_center"], v_center=g["v_center"])
        for k in ("k1", "k2", "k3", "p1", "p2", "l1", "l2", "l3"):
            setattr(m.precalib_params, k, g[k])
        m.set_model_params()
        m.units = "m"
        m.set_pose(np.asarray(F, float), np.eye(3))
        models.append(m)
    c = models[0].precalib_params.center_point
    gs = GUMStereo(models[0], models[1], center_point_top=c, center_point_top_inner=c, center_point_top_outer=c,
                   center_point_bottom=c, center_point_bottom_inner=c, center_point_bottom_outer=c,
                   radius_top_outer=rig.radii_top[1], radius_top_inner=rig.radii_top[0], radius_bottom_outer=rig.radii_bot[1],
                   radius_bottom_inner=rig.radii_bot[0])
    gs.set_current_omni_image(first_image, pano_width_in_pixels=pano_cols, generate_panoramas=True, view=False, apply_mask=True,
                              mask_RGB=(0, 0, 0))
    return gs


def golden_trajectory(n, seed):
    """Steady motion of 3-5 cm and 0.5-1.5 degrees per frame (every such frame passes run_VO's translation test and becomes a
    keyframe) with two nearly static frames in between (a few millimetres: they stay ordinary frames), so that the loop's
    keyframe branch, its no-keyframe branch and the pose chaining through the keyframe list are all exercised."""
    rng = np.random.default_rng(seed + 4242)
    T = np.eye(4)
    out = [T.copy()]
    for i in range(1, n):
        still = i in (3, 6)
        t = rng.normal(size=3)
        t[2] *= 0.3
        t = t / np.linalg.norm(t) * (rng.uniform(0.001, 0.003) if still else rng.uniform(0.03, 0.05))
        a = rng.normal(size=3)
        a /= np.linalg.norm(a)
        ang = np.deg2rad(rng.uniform(0.02, 0.1) if still else rng.uniform(0.5, 1.5))
        K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        S = np.eye(4)
        S[:3, :3] = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K
        S[:3, 3] = t
        T = T @ S
        out.append(T.copy())
    return np.array(out)


def main():
    import cv2
    install_extra_shims()
    from omnistereo import camera_models, pose_est_tools
    from vo_single_camera_sos_b200 import synth
    from .driver import quaternion_from_matrix

    rig = synth.make_rig(WIDTH, HEIGHT, PANO_COLS, seed=SEED)
    scene = synth.make_scene(N_LANDMARKS, seed=SEED)
    scene.half_extent = scene.half_extent * ROOM_SCALE    # a small room: 5-10 px of stereo disparity on this 800-px panorama
    traj = golden_trajectory(N_FRAMES, SEED)
    tmp = tempfile.mkdtemp(prefix="sos_vo_golden_")
    omni_dir = os.path.join(tmp, "omni")
    os.makedirs(omni_dir)
    images = [synth.render_omni(rig, scene, traj[i]) for i in range(N_FRAMES)]
    for i, img in enumerate(images):
        cv2.imwrite(os.path.join(omni_dir, "image-%06d.png" % i), img)
    gt_file = os.path.join(omni_dir, "gt_TUM.txt")
    with open(gt_file, "w") as f:
        for i in range(N_FRAMES):
            T = traj[i]
            q = quaternion_from_matrix(T)
            print(i, T[0, 3], T[1, 3], T[2, 3], q[1], q[2], q[3], q[0], file=f)
    gs = reference_gums(rig, PANO_COLS, images[0])

    # record what the reference's detector returns, call by call (top view then bottom view of every frame)
    recorded = []
    orig_detect = camera_models.OmniCamModel.detect_sparse_features_on_panorama

    def recording_detect(self, *a, **k):
        kp_list, desc_list = orig_detect(self, *a, **k)
        recorded.append((self.mirror_name, [cv2.KeyPoint_convert(list(kp)).reshape(-1, 2) if len(kp) else np.zeros((0, 2), np.float32) for kp in kp_list],
                         [np.zeros((0, 32), np.uint8) if d is None else np.asarray(d, np.uint8) for d in desc_list]))
        return kp_list, desc_list
    camera_models.OmniCamModel.detect_sparse_features_on_panorama = recording_detect

    results = os.path.join(tmp, "results")
    log = io.StringIO()
    with contextlib.redirect_stdout(log):
        pose_est_tools.run_VO(None, gs, gt_poses_filename=gt_file, est_poses_filename="estimated_frame_poses_TUM.txt",
                              img_filename_template=os.path.join(omni_dir, "image-*.png"), depth_filename_template=None,
                              img_indices=list(range(N_FRAMES)), results_path=results, thread_name="golden")
    camera_models.OmniCamModel.detect_sparse_features_on_panorama = orig_detect
    est = np.loadtxt(os.path.join(results, "estimated_frame_poses_TUM.txt"), ndmin=2)
    gt = np.loadtxt(os.path.join(results, "gt_associated_frame_poses_TUM.txt"), ndmin=2)
    keys = np.loadtxt(os.path.join(results, "keyframe_ids.txt"), ndmin=1).astype(np.int64)
    est_text = open(os.path.join(results, "estimated_frame_poses_TUM.txt")).read()
    assert est.shape == (N_FRAMES, 8), est.shape
    assert len(recorded) == 2 * N_FRAMES, len(recorded)

    out = dict(n_frames=np.int64(N_FRAMES), width=np.int64(WIDTH), height=np.int64(HEIGHT), pano_cols=np.int64(PANO_COLS),
               seed=np.int64(SEED), n_landmarks=np.int64(N_LANDMARKS), ransac_seed=np.int64(RANSAC_SEED),
               est_tum=est, gt_tum=gt, keyframe_ids=keys, est_tum_text=np.frombuffer(est_text.encode(), np.uint8),
               ransac_iterations=np.int64(210), trajectory=traj, room_scale=np.float64(ROOM_SCALE))
    tracker = pose_est_tools.TrackerStereoSE3(camera_model=gs, show_3D_points=False, save_correspondence_images=False,
                                              results_path=results)
    # the panorama geometry the reference derived from the model (rows, cylinder heights: it computes its own elevation limits
    # from the mirror radii, camera_models.py:1196-1382), needed to interpret the recorded panorama pixel coordinates
    for name, mdl in (("top", gs.top_model), ("bot", gs.bot_model)):
        pn = mdl.panorama
        out[f"pano_{name}"] = np.array([pn.cols, pn.rows, pn.pixel_size, pn.cyl_height_max, pn.cyl_circumference, pn.cyl_radius], np.float64)
        out[f"pano_{name}_cyl_height_min"] = np.float64(pn.z_height_min)
        out[f"elev_{name}"] = np.array([mdl.lowest_elevation_angle, mdl.highest_elevation_angle], np.float64)
    out["threshold"] = np.float64(tracker.backprojection_score_threshold_3D_to_2D)
    out["max_iterations"] = np.int64(tracker.max_ransac_iterations_3D_to_2D)
    out["max_horizontal_diff_f2f"] = np.float64(tracker.max_horizontal_diff_f2f_matches)
    out["cam_offsets"] = np.asarray(tracker.cam_offsets, np.float64)
    out["cam_rotations"] = np.asarray(tracker.cam_rotations, np.float64)
    assert len(RANSAC_CALLS) == N_FRAMES - 1
    for i, c in enumerate(RANSAC_CALLS, start=1):     # frame i was tracked with these arguments
        out[f"f{i}_ransac_points"], out[f"f{i}_ransac_bearings"], out[f"f{i}_ransac_cam"] = c["points"], c["bearings"], c["cam"]
        out[f"f{i}_ransac_best_hyp"], out[f"f{i}_ransac_inliers"], out[f"f{i}_ransac_pose"] = np.int64(c["best_hyp"]), c["inliers"], c["pose"]
    for i in range(N_FRAMES):
        for (name, kps, descs), view in zip(recorded[2 * i:2 * i + 2], ("top", "bot")):
            off = np.concatenate([[0], np.cumsum([len(k) for k in kps])]).astype(np.int32)
            out[f"f{i}_px_{view}"] = np.concatenate(kps).astype(np.float32) if off[-1] else np.zeros((0, 2), np.float32)
            out[f"f{i}_desc_{view}"] = np.concatenate(descs) if off[-1] else np.zeros((0, 32), np.uint8)
            out[f"f{i}_boff_{view}"] = off
    np.savez_compressed(os.path.join(OUT, "vo_sequence.npz"), **out)
    shutil.rmtree(tmp, ignore_errors=True)
    print(f"vo_sequence.npz: {N_FRAMES} frames, keyframes {keys.tolist()}, "
          f"features/view ~{int(np.mean([len(out[f'f{i}_px_top']) for i in range(N_FRAMES)]))}, "
          f"end position error {np.linalg.norm(est[-1, 1:4] - gt[-1, 1:4]):.4f} m")
    print(log.getvalue()[-600:])


if __name__ == "__main__":
    main()
