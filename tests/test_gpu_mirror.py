"""GPU: the host-side mirror of the reference interface (omnistereo.* / pyopengv) against the golden vectors that the
reference's own classes produced for the same inputs (oracle/gen_golden.py).  These read like the reference's tests
would: same class names, same method names, same keyword arguments."""
import pickle

import cv2
import numpy as np
import pytest

from conftest import load_golden, sub
from oracle import gft as ogft

pytestmark = pytest.mark.gpu


def build_gums(g):
    """The synthetic GUMS of oracle/gen_golden.py::build_gums, rebuilt through the mirrored constructors."""
    from omnistereo.gum import GUM, GUMStereo
    W, H = 320, 240
    models = []
    for name, z_axis, F in (("top", 1.0, [0, 0, 0.12]), ("bot", -1.0, [0, 0, 0])):
        p = sub(g, f"gum_{name}_")
        m = GUM(precalib_filename="/nonexistent", new_method=True, z_axis=z_axis, image_size_pixels=(W, H),
                center_uv_point=(p["u_center"], p["v_center"]))
        m.precalib_params.set_gum_params(xi1=p["xi1"], xi2=p["xi2"], xi3=p["xi3"])
        m.precalib_params.set_generalized_cam_params(gamma1=p["gamma1"], gamma2=p["gamma2"], alpha_c=p["alpha_c"],
                                                     u_center=p["u_center"], v_center=p["v_center"])
        for k in ("k1", "k2", "k3", "p1", "p2", "l1", "l2", "l3"):
            setattr(m.precalib_params, k, p[k])
        m.set_model_params()
        m.units = "m"
        m.set_pose(np.array(F, float), np.eye(3))
        models.append(m)
    c = models[0].precalib_params.center_point
    gs = GUMStereo(models[0], models[1], center_point_top=c, center_point_top_inner=c, center_point_top_outer=c,
                   center_point_bottom=c, center_point_bottom_inner=c, center_point_bottom_outer=c,
                   radius_top_outer=0.48 * H, radius_top_inner=0.30 * H, radius_bottom_outer=0.28 * H,
                   radius_bottom_inner=0.08 * H)
    # The mirror estimates the elevation bounds with the closed-form lifting; the reference runs a per-pixel optimisation
    # of the forward projection for this one-off set-up step (camera_models.py:1196-1382, out of scope, SURVEY §2 row 5).
    # They agree to a few mrad; a calibrated model carries the reference's values, so install those:
    for name, m in (("top", gs.top_model), ("bot", gs.bot_model)):
        lo, hi = g[f"elev_{name}"]
        assert abs(m.lowest_elevation_angle - lo) < 5e-3 and abs(m.highest_elevation_angle - hi) < 5e-3
        m.lowest_elevation_angle, m.highest_elevation_angle = float(lo), float(hi)
    glo = min(gs.top_model.lowest_elevation_angle, gs.bot_model.lowest_elevation_angle)
    ghi = max(gs.top_model.highest_elevation_angle, gs.bot_model.highest_elevation_angle)
    for m in (gs.top_model, gs.bot_model):
        m.globally_lowest_elevation_angle, m.globally_highest_elevation_angle = glo, ghi
    return gs


@pytest.fixture(scope="module")
def gums(ctx):
    g = load_golden("remap.npz")
    gs = build_gums(g)
    gs.set_current_omni_image(g["img"], pano_width_in_pixels=200, generate_panoramas=True, view=False, apply_mask=True,
                              mask_RGB=(0, 0, 0))
    return gs, g


def test_set_current_omni_image_gives_the_reference_panoramas(gums):
    gs, g = gums
    for name, m in (("top", gs.top_model), ("bot", gs.bot_model)):
        p = m.panorama
        assert (p.rows, p.cols) == g[f"pano_{name}"].shape[:2]
        assert np.array_equal(m.mask, g[f"mask_{name}"])
        ok = ~np.isnan(g[f"map_x32_{name}"])
        assert np.array_equal(np.isnan(p.world2cam_LUT_map_x), ~ok)
        assert np.max(np.abs(p.world2cam_LUT_map_x[ok] - g[f"map_x32_{name}"][ok])) < 1 / 64
        # the mirrored LUT differs from the reference's by < 1/64 px (the reference evaluates parts in float32), which can
        # move a Q5 coordinate by one step; with the REFERENCE's LUT the remap is bit-exact:
        p.world2cam_LUT_map_x = g[f"map_x32_{name}"].astype(np.float64)
        p.world2cam_LUT_map_y = g[f"map_y32_{name}"].astype(np.float64)
    gs.set_current_omni_image(g["img"], generate_panoramas=False, view=False, apply_mask=True, mask_RGB=(0, 0, 0))
    assert np.array_equal(gs.top_model.panorama.panoramic_img, g["pano_top"])
    assert np.array_equal(gs.bot_model.panorama.panoramic_img, g["pano_bot"])
    masked_top, _ = gs.get_fully_masked_images(omni_img=g["img"], view=False, color_RGB=(10, 200, 90))
    out = gs.top_model.panorama.get_panoramic_image(masked_top, set_own=False, border_RGB_color=(30, 60, 250))
    assert np.array_equal(out, g["pano_colour_top"])
    out = gs.top_model.panorama.get_panoramic_image(gs.top_model.mask, set_own=False, border_RGB_color=(0, 0, 0))
    assert np.array_equal(out, g["pano_of_mask_top"])


def test_feature_matcher_match(ctx):
    from omnistereo.camera_models import FeatureMatcher
    g = load_golden("hamming.npz")
    m = FeatureMatcher("ORB", "BF", 1, percentage_good_matches=1.0).match(query_descriptors=g["q"], train_descriptors=g["t"])
    assert isinstance(m[0], cv2.DMatch)
    assert [x.queryIdx for x in m] == g["nn_q"].tolist() and [x.trainIdx for x in m] == g["nn_t"].tolist()
    assert [x.distance for x in m] == g["nn_d"].tolist()
    fm = FeatureMatcher("ORB", "BF", 1, cross_check=True)
    qi, ti, dd = fm.match_arrays(g["q"], g["t"])
    order = np.argsort(qi, kind="stable")
    assert np.array_equal(qi[order], g["cross_q"]) and np.array_equal(ti[order], g["cross_t"])
    assert FeatureMatcher("ORB", "BF", 1).match(np.zeros((0, 32), np.uint8), g["t"]) == []
    with pytest.raises(NotImplementedError):
        FeatureMatcher("ORB", "BF", 3)


def test_feature_matcher_k_best_2_on_binary_descriptors(ctx):
    """camera_models.py:417-444: for ORB the k_best = 2 branch keeps BOTH neighbours of every query (the Lowe ratio test
    is SIFT-only), flattens query by query and sorts stably by distance.  Golden from the reference's own class."""
    from omnistereo.camera_models import FeatureMatcher
    g = load_golden("hamming.npz")
    m = FeatureMatcher("ORB", "BF", 2).match(query_descriptors=g["q"], train_descriptors=g["t"])
    assert len(m) == 2 * len(g["q"])
    assert [x.queryIdx for x in m] == g["k2_q"].tolist() and [x.trainIdx for x in m] == g["k2_t"].tolist()
    assert [x.distance for x in m] == g["k2_d"].tolist()
    # a single train row gives one neighbour per query
    m1 = FeatureMatcher("ORB", "BF", 2).match(query_descriptors=g["q"][:5], train_descriptors=g["t"][:1])
    assert len(m1) == 5 and all(x.trainIdx == 0 for x in m1)
    # the explicit (non-reference) ratio kwarg still selects the Lowe test on the device
    from oracle import hamming
    qi, ti, dd = FeatureMatcher("ORB", "BF", 2, ratio=0.75).match_arrays(g["q"], g["t"])
    oq, ot, od = hamming.match_select(g["q"], g["t"], "ratio", ratio=0.75)
    assert np.array_equal(qi, oq) and np.array_equal(ti, ot) and np.array_equal(dd, od)


def test_feature_matcher_radius_match(ctx):
    """use_radius_match=True (camera_models.py:409-412): goldens from the reference's own class at an integer and a fractional
    descriptor radius, plus a dense case against the oracle (many rows per query, ties within a query)."""
    from omnistereo.camera_models import FeatureMatcher
    from oracle import hamming
    g = load_golden("hamming.npz")
    fm = FeatureMatcher("ORB", "BF", 1, use_radius_match=True)
    for tag in ("r40", "r70"):
        m = fm.match(query_descriptors=g["q"], train_descriptors=g["t"], max_descriptor_distance_radius=float(g[f"{tag}_radius"]))
        assert [x.queryIdx for x in m] == g[f"{tag}_q"].tolist() and [x.trainIdx for x in m] == g[f"{tag}_t"].tolist()
        assert [x.distance for x in m] == g[f"{tag}_d"].tolist()
    rng = np.random.default_rng(4)
    q = rng.integers(0, 256, (333, 32), dtype=np.uint8)
    t = rng.integers(0, 256, (517, 32), dtype=np.uint8)
    qi, ti, dd = fm.match_arrays(q, t, max_descriptor_distance_radius=118)
    oq, ot, od = hamming.radius_match_flat_sorted(q, t, 118)
    assert len(oq) > 5000 and np.array_equal(qi, oq) and np.array_equal(ti, ot) and np.array_equal(dd, od)
    assert fm.match(q, t, max_descriptor_distance_radius=20) == []


def test_stereo_and_temporal_matching(gums):
    from omnistereo import pose_est_tools
    from omnistereo.camera_models import FeatureMatcher
    gs, _ = gums
    g = load_golden("matching_frames.npz")
    gs.feature_matcher_for_static_stereo = FeatureMatcher("ORB", "BF", 1, percentage_good_matches=1.0)
    gs.feature_matcher_for_motion = FeatureMatcher("ORB", "BF", 1, percentage_good_matches=1.0)
    nb = int(g["n_buckets"])
    kp = lambda pts: [cv2.KeyPoint(float(x), float(y), 7.0) for x, y in pts]
    (m_top, k_top, d_top), (m_bot, k_bot, d_bot), colors = gs.match_features_panoramic_top_bottom(
        keypts_list_top=[kp(g[f"b{b}_pt_top"]) for b in range(nb)], desc_list_top=[g[f"b{b}_d_top"] for b in range(nb)],
        keypts_list_bot=[kp(g[f"b{b}_pt_bot"]) for b in range(nb)], desc_list_bot=[g[f"b{b}_d_bot"] for b in range(nb)],
        min_rectified_disparity=1, max_horizontal_diff=2.5, show_matches=False)
    assert np.array_equal(m_top, g["stereo_m_top"]) and np.array_equal(m_bot, g["stereo_m_bot"])
    assert np.array_equal(d_top, g["stereo_desc_top"]) and np.array_equal(d_bot, g["stereo_desc_bot"])
    assert len(colors) == len(m_top) and k_top[0].pt == (m_top[0, 0], m_top[0, 1])
    kq = np.array(kp(g["f2f_pq"][:, :2])); kt = np.array(kp(g["f2f_pt"][:, :2]))
    (ti, ktm, dtm), (qi, kqm, dqm), _ = pose_est_tools.match_features_frame_to_frame(
        cam_model=gs, train_kpts=kt, train_desc=g["f2f_t"], query_kpts=kq, query_desc=g["f2f_q"],
        random_colors_RGB=np.zeros((len(kt), 3), np.uint8), max_horizontal_diff=float(g["f2f_max_du"]),
        keypts_as_points_train=g["f2f_pt"], keypts_as_points_query=g["f2f_pq"])
    assert np.array_equal(ti, g["f2f_train_idx"]) and np.array_equal(qi, g["f2f_query_idx"])
    assert np.array_equal(dtm, g["f2f_t"][ti])


def test_lifting_triangulation_and_gates(gums):
    from omnistereo.common_cv import filter_pixel_correspondences
    gs, _ = gums
    g = load_golden("lifting.npz")
    top = gs.top_model
    az, el = top.panorama.get_direction_angles_from_pixel_pano(g["pano_px"], use_LUTs=False)
    assert np.allclose(az, g["pano_az"], rtol=0, atol=1e-12, equal_nan=True)
    assert np.allclose(el, g["pano_el"], rtol=0, atol=1e-12, equal_nan=True)
    b = top.get_3D_point_from_angles_wrt_focus(azimuth=az, elevation=el)
    assert b.shape == (1, len(az), 4) and np.allclose(b[0, :, :3], g["pano_bearing"], atol=1e-12, equal_nan=True)
    xyz = gs.get_triangulated_point_from_direction_angles(dir_angs_top=(g["tri_az1"], g["tri_el1"]),
                                                          dir_angs_bot=(g["tri_az2"], g["tri_el2"]),
                                                          use_midpoint_triangulation=True)
    assert xyz.shape == (1, len(g["tri_az1"]), 4)
    assert np.allclose(xyz[0], g["tri_xyz_homo"], rtol=1e-9, atol=1e-11)
    assert np.array_equal(gs.filter_panoramic_points_due_to_range(xyz[0], min_3D_range=0.5, max_3D_range=7.0), g["tri_valid_homo"])
    assert np.array_equal(gs.filter_panoramic_points_due_to_range(xyz[0][:, :3], min_3D_range=0.5, max_3D_range=7.0), g["tri_valid_xyz"])
    for name, m in (("top", gs.top_model), ("bot", gs.bot_model)):
        pre = f"heik_{name}_"
        Ps = m.lift_pixel_to_unit_sphere_wrt_focus(g[pre + "omni_uv"][None])
        assert np.allclose(Ps[0], g[pre + "sphere"], rtol=1e-7, atol=1e-10)
        a, e = m.get_direction_angles_from_pixel(g[pre + "omni_uv"][None])
        assert np.allclose(a[0], g[pre + "omni_az"], atol=1e-9) and np.allclose(e[0], g[pre + "omni_el"], atol=1e-9)
        P = np.hstack([g[pre + "proj_pts"], np.ones((len(g[pre + "proj_pts"]), 1))])[None]
        u, v, mh = m.get_pixel_from_3D_point_wrt_M(P)
        assert np.allclose(u[0], g[pre + "proj_u"], rtol=1e-9) and np.allclose(v[0], g[pre + "proj_v"], rtol=1e-9)
        assert mh.shape == (1, P.shape[1], 3)
    ok = filter_pixel_correspondences(np.array([[10.0, 5.0], [10.0, 5.0], [13.0, 9.0]]), np.array([[12.5, 4.0], [12.6, 4.0], [13.0, 8.5]]), 1, 2.5)
    assert ok.tolist() == [True, False, False]


def test_rgbd_model_and_superimposition(ctx):
    from omnistereo.camera_models import RGBDCamModel
    from omnistereo.transformations import superimposition_matrix
    g = load_golden("rgbd.npz")
    for tag, kw in (("z", dict(fx=52.5, fy=52.5, center_x=31.5, center_y=23.5, depth_is_Z=True)),
                    ("radial", dict(fx=55.4256258, fy=55.4256258, center_x=31.5, center_y=23.5, depth_is_Z=False,
                                    focal_length_m=1.0 / 1000.0))):
        cam = RGBDCamModel(**kw)
        xyz = cam.get_XYZ(depth=g["depth"], u_coords=g["u"].astype(np.uint), v_coords=g["v"].astype(np.uint))
        assert xyz.shape == (1, len(g["u"]), 3)
        assert np.allclose(xyz[0], g[f"{tag}_xyz"], rtol=1e-4, atol=1e-7, equal_nan=True)
        assert np.allclose(cam.get_depth_Z(g["depth"]), g[f"{tag}_depth_z"], rtol=1e-4)
    a = load_golden("arun.npz")
    for k in (3, 4, 100):
        M = superimposition_matrix(a[f"k{k}_v0"][0].T, a[f"k{k}_v1"][0].T, scale=False, usesvd=True)
        assert M.shape == (4, 4) and np.allclose(M[:3], a[f"k{k}_M"][0], atol=1e-9) and np.allclose(M[3], [0, 0, 0, 1])
    # Umeyama: recover a similarity transform
    rng = np.random.default_rng(0)
    v0 = rng.normal(size=(3, 50))
    R = a["k3_M"][0][:, :3]
    v1 = 1.7 * R @ v0 + np.array([[0.3], [-0.2], [0.9]])
    M = superimposition_matrix(v0, v1, scale=True)
    assert np.allclose(M[:3, :3], 1.7 * R, atol=1e-9) and np.allclose(M[:3, 3], [0.3, -0.2, 0.9], atol=1e-9)


def test_trackers_on_a_synthetic_pair(gums):
    """StereoPanoramicFrame + TrackerStereoSE3.track_frame end to end on synthetic features with a known motion."""
    import pyopengv
    from omnistereo import pose_est_tools
    from vo_single_camera_sos_b200 import synth
    gs, _ = gums
    assert pyopengv.absolute_pose_noncentral_ransac is pose_est_tools.absolute_pose_noncentral_ransac
    tracker = pose_est_tools.TrackerStereoSE3(gs)
    assert tracker.max_ransac_iterations_3D_to_2D == 210
    assert abs(tracker.backprojection_score_threshold_3D_to_2D - (1 - np.cos(np.deg2rad(5)))) < 1e-15
    pano = gs.top_model.panorama
    rig = synth.Rig(320, 240, {}, {}, gs.top_model.F[:3, 0].copy(), gs.bot_model.F[:3, 0].copy(),
                    (gs.top_model.lowest_elevation_angle, gs.top_model.highest_elevation_angle),
                    (gs.bot_model.lowest_elevation_angle, gs.bot_model.highest_elevation_angle), (0, 0), (0, 0), pano.cols,
                    dict(cols=pano.cols, rows=pano.rows, pixel_size=pano.pixel_size, cyl_height_max=pano.cyl_height_max,
                         cyl_height_min=pano.z_height_min, cyl_circumference=pano.cyl_circumference, cyl_radius=1.0))
    # this test rig has disjoint elevation bands (SURVEY §8c) -> widen both to the panorama so landmarks are co-visible
    rig.elev_top = rig.elev_bot = (pano.globally_lowest_elevation_angle + 1e-3, pano.globally_highest_elevation_angle - 1e-3)
    scene = synth.make_scene(1500, seed=2)
    traj = synth.make_trajectory(2, seed=4)
    frames = []
    for i in range(2):
        f = synth.make_frame_features(rig, scene, traj[i], 600, 12, seed=50 + i, cap=600, px_sigma=0.02)
        lists = []
        for which in ("top", "bot"):
            off = f[which]["bucket_off"]
            lists.append([[cv2.KeyPoint(float(x), float(y), 7.0) for x, y in f[which]["px"][off[k]:off[k + 1]]] for k in range(12)])
            lists.append([f[which]["desc"][off[k]:off[k + 1]] for k in range(12)])
        frames.append(pose_est_tools.StereoPanoramicFrame(gs, i, features=tuple(lists)))
        assert frames[-1].num_valid_keypoints > 50
        pc = frames[-1].pano_correspondences
        assert pc.points_3D_coords_homo.shape == (frames[-1].num_valid_keypoints, 4) and pc.m_top.shape[1] == 3
    ok, msg = tracker.track_frame(frames[0], frames[1])
    assert ok, msg
    T_rel = np.linalg.inv(traj[0]) @ traj[1]
    T = frames[1].T_frame_wrt_tracking_ref_frame
    assert tracker.num_tracked_correspondences > 30
    assert np.allclose(T[:3, :3], T_rel[:3, :3], atol=0.05) and np.allclose(T[:3, 3], T_rel[:3, 3], atol=0.25)  # 200-px panorama: 1.8 deg per pixel
    # models with lazily built device state survive a pickle round trip (demo_vo_sos.py:109 loads a pickled GUMStereo)
    gs2 = pickle.loads(pickle.dumps(gs))
    assert np.array_equal(gs2.top_model.panorama.world2cam_LUT_map_x, gs.top_model.panorama.world2cam_LUT_map_x, equal_nan=True)


def test_detect_sparse_features_gft_on_device(gums):
    """OmniCamModel.detect_sparse_features_on_panorama(feature_detection_method="GFT", median_win_size=11) — the
    reference's default detector (pose_est_tools.py:681, 297) — against the reference's own call sequence made with cv2:
    medianBlur -> BGR2GRAY -> goodFeaturesToTrack per azimuthal mask -> KeyPoint_convert -> ORB.compute
    (camera_models.py:1706-1768)."""
    gs, _ = gums
    rng = np.random.default_rng(11)
    for model in (gs.top_model, gs.bot_model):
        pano_obj = model.panorama
        rows, cols = pano_obj.rows, pano_obj.cols
        # a textured panorama large enough for ORB's 31-pixel border (the golden rig's own panorama is 48 rows high)
        pano = cv2.GaussianBlur(rng.integers(0, 256, (160, 480, 3), dtype=np.uint8), (0, 0), 1.6)
        masks = []
        for k in range(4):
            m = np.zeros(pano.shape[:2], np.uint8)
            m[8:-8, k * 120:(k + 1) * 120] = 255
            masks.append(m)
        saved = pano_obj.panoramic_img, pano_obj.azimuthal_masks
        pano_obj.panoramic_img, pano_obj.azimuthal_masks = pano, masks
        try:
            kl, dl = model.detect_sparse_features_on_panorama(feature_detection_method="GFT", num_of_features=60,
                                                              median_win_size=11, show=False)
        finally:
            pano_obj.panoramic_img, pano_obj.azimuthal_masks = saved
        blurred = cv2.cvtColor(cv2.medianBlur(pano, 11), cv2.COLOR_BGR2GRAY)
        orb = cv2.ORB_create(nfeatures=60)
        eig = ogft.corner_min_eigenval(blurred)
        total = same = 0
        for m, k_got, d_got in zip(masks, kl, dl):
            # exactly: cv2 median and gray, then the oracle's Shi-Tomasi, then ORB.compute
            want, _ = ogft.good_features(eig, m, 60, 0.01, 5.0)
            k_or, d_or = orb.compute(blurred, list(cv2.KeyPoint_convert(want)))
            assert [k.pt for k in k_got] == [k.pt for k in k_or] and np.array_equal(d_got, d_or)
            # against cv2's own corner lists (its SIMD tail columns may decide a near-tie differently)
            pts = cv2.goodFeaturesToTrack(image=blurred, maxCorners=60, qualityLevel=0.01, minDistance=5, mask=m,
                                          useHarrisDetector=False)
            k_ref, d_ref = orb.compute(blurred, list(cv2.KeyPoint_convert(pts.reshape(-1, 2))))
            assert abs(len(k_got) - len(k_ref)) <= 1 and d_got.shape[1] == 32
            n = min(len(k_got), len(k_ref))
            for a, b, da, db in zip(k_got[:n], k_ref[:n], d_got[:n], d_ref[:n]):
                total += 1
                if a.pt == b.pt:
                    same += 1
                    assert np.array_equal(da, db) and a.angle == b.angle == -1 and a.octave == b.octave == 0
        assert total > 60 and same >= 0.98 * total, (same, total)


def test_detect_sparse_features_gft_refuses_overflow(gums):
    """Without azimuthal masks the whole panorama is one list; a textured 849 x 2400 panorama has far more than the 16 384
    candidates the selection can rank, and the call raises instead of returning fewer keypoints."""
    from vo_single_camera_sos_b200._lib import SosError
    gs, _ = gums
    pano = cv2.GaussianBlur(np.random.default_rng(12).integers(0, 256, (849, 2400, 3), dtype=np.uint8), (0, 0), 1.0)
    gray = cv2.cvtColor(cv2.medianBlur(pano, 11), cv2.COLOR_BGR2GRAY)
    assert len(ogft.candidates(ogft.corner_min_eigenval(gray), None, 0.01)) > 16384
    pano_obj = gs.top_model.panorama
    saved = pano_obj.panoramic_img, pano_obj.azimuthal_masks
    pano_obj.panoramic_img, pano_obj.azimuthal_masks = pano, []
    try:
        with pytest.raises(SosError):
            gs.top_model.detect_sparse_features_on_panorama(feature_detection_method="GFT", num_of_features=60,
                                                            median_win_size=11, show=False)
    finally:
        pano_obj.panoramic_img, pano_obj.azimuthal_masks = saved
