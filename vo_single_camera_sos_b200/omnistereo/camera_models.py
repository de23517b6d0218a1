"""Mirror of the hot-path classes of omnistereo/camera_models.py (SURVEY §2 rows 2, 4-7)."""
import cv2
import numpy as np
import torch

from . import device_context, to_device
from .. import ops


def get_normalized_points(points_wrt_M):
    """camera_models.py:203-212 (host glue on a few thousand points)."""
    p = np.asarray(points_wrt_M, np.float64)
    return p[..., :3] / (np.linalg.norm(p[..., :3], axis=-1)[..., np.newaxis])


# ---------------------------------------------------------------------------------------------------------------------
# F4: the matcher (camera_models.py:364-446)
# ---------------------------------------------------------------------------------------------------------------------
class FeatureMatcher(object):
    """Brute-force descriptor matcher with the reference's interface.  For binary descriptors ("ORB", ...) the distances
    are Hamming distances computed by sos_hamming_top2; results are ordered like sorted(matches, key=distance), i.e.
    stably by (distance, queryIdx), with ties between train rows going to the lowest trainIdx (cv2.BFMatcher).
    method "SIFT" / "SURF" selects the L2 norm on float descriptors like the reference (camera_models.py:397-399): the
    tensor-core matcher sos_l2_top2 for integer-valued descriptors in [0, 255] (cv2's SIFT output, exact), sos_l2f_top2 for
    any other finite values (SURF, KAZE, RootSIFT: bit-equal to a float64 reference)."""

    def __init__(self, method, matcher_type, k_best, *args, **kwargs):
        self.feature_detection_method = method
        self.matcher_type = matcher_type
        self.k_best = k_best
        self.MIN_MATCH_COUNT = 10
        self.percentage_good_matches = kwargs.get("percentage_good_matches", 1.0)
        self.num_of_features = kwargs.get("num_of_features", 100)
        self.use_radius_match = kwargs.get("use_radius_match", False)
        self.cross_check = kwargs.get("cross_check", False)   # BFMatcher(crossCheck=True), commented out at :401
        # Lowe's ratio test exists in the reference only for method == "SIFT" with k_best == 2 (:421-436, ratio 0.75);
        # a "ratio" kwarg (not in the reference) requests it explicitly for binary descriptors.
        self.ratio = kwargs.get("ratio", None)
        if matcher_type != "BF":
            raise NotImplementedError("only the brute-force matcher of the reference's default path is mirrored")
        self.float_descriptors = str(method).upper() in ("SIFT", "SURF")
        if self.float_descriptors and (self.use_radius_match or self.cross_check):
            raise NotImplementedError("radius match / cross check are mirrored for binary descriptors only")
        if self.k_best > 2:
            raise NotImplementedError("k_best > 2 is not mirrored (the device kernel keeps the two nearest neighbours)")

    def match_arrays(self, query_descriptors, train_descriptors, max_descriptor_distance_radius=-1, px_query=None,
                     px_train=None, max_horizontal_diff=-1.0, min_rectified_disparity=-1.0):
        """(queryIdx, trainIdx, distance) int32 arrays in the reference's output order; optional fused pixel gate."""
        if self.float_descriptors:
            return self._match_arrays_l2(query_descriptors, train_descriptors, px_query, px_train, max_horizontal_diff,
                                         min_rectified_disparity)
        q = np.ascontiguousarray(query_descriptors, np.uint8)
        t = np.ascontiguousarray(train_descriptors, np.uint8)
        if q.ndim != 2 or t.ndim != 2 or q.shape[1] != 32 or t.shape[1] != 32:
            raise ValueError("descriptors must be N x 32 uint8 (256-bit)")
        nq, nt = len(q), len(t)
        empty = np.zeros(0, np.int32)
        if nq == 0 or nt == 0:
            return empty, empty, empty
        ctx = device_context()
        if self.use_radius_match:
            # camera_models.py:409-412: radiusMatch (every train row within the descriptor distance), flattened query by
            # query, then sorted(key=distance) — stable.  cv2 compares float distances: d <= maxDistance.
            qi, ti, dd = ctx.hamming_radius(to_device(q), to_device(t), int(np.floor(max_descriptor_distance_radius)))
            qi, ti, dd = qi.cpu().numpy().astype(np.int32), ti.cpu().numpy(), dd.cpu().numpy()
            within = np.lexsort((ti, dd, qi))            # per query by (distance, train index): cv2 sorts each query's list
            qi, ti, dd = qi[within], ti[within], dd[within]
            order = np.argsort(dd, kind="stable")
            qi, ti, dd = qi[order], ti[order], dd[order]
            if px_query is not None and px_train is not None:
                from .common_cv import filter_pixel_correspondences
                ok = filter_pixel_correspondences(np.asarray(px_train)[ti], np.asarray(px_query)[qi],
                                                  min_rectified_disparity, max_horizontal_diff)
                qi, ti, dd = qi[ok], ti[ok], dd[ok]
            return qi, ti, dd
        dev = ctx.device
        i32 = lambda v: torch.tensor([v], dtype=torch.int32, device=dev)
        zero, nq_d, nt_d = i32(0), i32(nq), i32(nt)
        qd, td = to_device(q), to_device(t)
        i0, d0, i1, d1 = ctx.hamming_top2(qd, td, zero, nq_d, zero, nt_d, nq, nt, want_second=True)
        gate = px_query is not None and px_train is not None
        if self.k_best == 2 and not self.cross_check and self.ratio is None:
            # camera_models.py:417-444 for binary descriptors: knnMatch(k=2) flattened query by query (both neighbours
            # kept, no ratio test), then sorted(key=distance) — stable, so ties keep the (query, neighbour rank) order.
            i0, d0, i1, d1 = (x.cpu().numpy() for x in (i0, d0, i1, d1))
            qi = np.repeat(np.arange(nq, dtype=np.int32), 2)
            ti = np.stack([i0, i1], 1).reshape(-1)
            dd = np.stack([d0, d1], 1).reshape(-1)
            have = ti >= 0                                   # a train set of one row yields one neighbour per query
            qi, ti, dd = qi[have], ti[have], dd[have]
            order = np.argsort(dd, kind="stable")
            qi, ti, dd = qi[order], ti[order], dd[order]
            if gate:
                from .common_cv import filter_pixel_correspondences
                ok = filter_pixel_correspondences(np.asarray(px_train)[ti], np.asarray(px_query)[qi],
                                                  min_rectified_disparity, max_horizontal_diff)
                qi, ti, dd = qi[ok], ti[ok], dd[ok]
            return qi, ti.astype(np.int32), dd.astype(np.int32)
        mode, rev = ops.MATCH_NN, None
        if self.cross_check:
            mode = ops.MATCH_CROSS
            rev = ctx.hamming_top2(td, qd, zero, nt_d, zero, nq_d, nt, nq, want_second=False)[0]
        elif self.k_best == 2 and self.ratio is not None and self.ratio > 0:
            mode = ops.MATCH_RATIO
        oq, ot, od, oc = ctx.match_select(
            mode, i0, d0, d1, zero, nq_d, zero, rev_idx0=rev,
            px_q=to_device(np.asarray(px_query)[:, :2], torch.float32) if gate else None,
            px_t=to_device(np.asarray(px_train)[:, :2], torch.float32) if gate else None,
            max_du=float(max_horizontal_diff), min_dv=float(min_rectified_disparity), ratio=float(self.ratio or 0.75))
        n = int(oc.cpu().numpy()[0])
        return oq[:n].cpu().numpy(), ot[:n].cpu().numpy(), od[:n].cpu().numpy()

    def _match_arrays_l2(self, query_descriptors, train_descriptors, px_query, px_train, max_du, min_dv):
        """The SIFT / SURF branch (camera_models.py:397-399, 417-442): cv2.BFMatcher() = NORM_L2.  k_best = 1: the nearest
        train row per query; k_best = 2: knnMatch(k = 2), for "SIFT" filtered by Lowe's ratio test m0.distance <
        0.75 * m1.distance (len(m) == 2 required, :423), otherwise both neighbours flattened; then sorted(key=distance).
        Distances are float32 like cv2's.  The engine follows the values: integers in [0, 255] go to l2_top2 (9 MMAs per
        tile pair, no re-decision), everything else to l2f_top2 (13 to 25 MMAs and a float64 decision)."""
        q = np.ascontiguousarray(query_descriptors, np.float32)
        t = np.ascontiguousarray(train_descriptors, np.float32)
        if q.ndim != 2 or t.ndim != 2 or q.shape[1] != t.shape[1] or q.shape[1] > 128:
            raise ValueError("float descriptors must be N x dim float32 with dim <= 128")
        nq, nt = len(q), len(t)
        if nq == 0 or nt == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32)
        ctx = device_context()
        i32 = lambda v: torch.tensor([v], dtype=torch.int32, device=ctx.device)
        zero = i32(0)
        integer = all(np.array_equal(x, np.floor(x)) and x.min() >= 0 and x.max() <= 255 for x in (q, t))
        top2 = ctx.l2_top2 if integer else ctx.l2f_top2
        i0, d0, i1, d1 = (x.cpu().numpy() for x in top2(to_device(q), to_device(t), zero, i32(nq), zero, i32(nt), nq, nt))
        qi = np.arange(nq, dtype=np.int32)
        if self.k_best == 2 and str(self.feature_detection_method).upper() == "SIFT":
            keep = (i1 >= 0) & (d0.astype(np.float64) < d1.astype(np.float64) * 0.75)      # Python floats in the reference
            qi, ti, dd = qi[keep], i0[keep], d0[keep]
        elif self.k_best == 2:
            qi = np.repeat(qi, 2)
            ti, dd = np.stack([i0, i1], 1).reshape(-1), np.stack([d0, d1], 1).reshape(-1)
            have = ti >= 0
            qi, ti, dd = qi[have], ti[have], dd[have]
        else:
            ti, dd = i0, d0
        order = np.argsort(dd, kind="stable")
        qi, ti, dd = qi[order], ti[order], dd[order]
        if px_query is not None and px_train is not None:
            from .common_cv import filter_pixel_correspondences
            ok = filter_pixel_correspondences(np.asarray(px_train)[ti], np.asarray(px_query)[qi], min_dv, max_du)
            qi, ti, dd = qi[ok], ti[ok], dd[ok]
        return qi, ti.astype(np.int32), dd

    def match(self, query_descriptors, train_descriptors, max_descriptor_distance_radius=-1):
        """List of cv2.DMatch sorted by distance — the reference's return type (camera_models.py:404-446)."""
        qi, ti, dd = self.match_arrays(query_descriptors, train_descriptors, max_descriptor_distance_radius)
        return [cv2.DMatch(int(a), int(b), float(c)) for a, b, c in zip(qi, ti, dd)]


# ---------------------------------------------------------------------------------------------------------------------
# T1: correspondence containers (camera_models.py:250-362)
# ---------------------------------------------------------------------------------------------------------------------
def _flatten(list_of_lists):
    out = []
    for x in list_of_lists:
        if x is not None:
            out.extend(list(x))
    return out


class KeyPointAndDescriptor(object):
    def __init__(self, kpts_list, desc_list, coords_array=None, random_colors_RGB_list=[], do_flattening=False, **kwargs):
        if do_flattening:
            self.keypoints = _flatten(kpts_list)
            self.descriptors = np.array(_flatten(desc_list))
        else:
            self.keypoints = kpts_list
            self.descriptors = desc_list
        l = len(self.keypoints)
        if coords_array is None or len(coords_array) == 0:
            self.pixel_coords = np.ones((1, l, 3))
            for idx in range(l):
                self.pixel_coords[0, idx, 0] = self.keypoints[idx].pt[0]
                self.pixel_coords[0, idx, 1] = self.keypoints[idx].pt[1]
        else:
            self.pixel_coords = coords_array
        if random_colors_RGB_list is None or len(random_colors_RGB_list) < l:
            self.random_colors_RGB = np.random.randint(low=0, high=256, size=(l, 3), dtype="uint8")
        else:
            self.random_colors_RGB = random_colors_RGB_list


class PanoramicCorrespondences(object):
    def __init__(self, kpts_top_list, desc_top_list, kpts_bot_list, desc_bot_list, points_3D=None, m_top_array=None,
                 m_bot_array=None, random_colors_RGB_list=[], do_flattening=False, **kwargs):
        if do_flattening:
            self.kpts_top, self.kpts_bot = _flatten(kpts_top_list), _flatten(kpts_bot_list)
            self.desc_top, self.desc_bot = np.array(_flatten(desc_top_list)), np.array(_flatten(desc_bot_list))
        else:
            self.kpts_top, self.kpts_bot = kpts_top_list, kpts_bot_list
            self.desc_top, self.desc_bot = desc_top_list, desc_bot_list
        if points_3D is not None:
            if len(points_3D) > 0:
                if points_3D.shape[-1] == 3:
                    self.points_3D_coords_homo = np.ones((len(points_3D), 4))
                    self.points_3D_coords_homo[:, :3] = points_3D[:, :3]
                else:
                    self.points_3D_coords_homo = points_3D
            else:
                self.points_3D_coords_homo = np.empty((0, 4))
        else:
            self.points_3D_coords_homo = []

        def homo(kpts, arr):
            if arr is not None and len(arr) > 0:
                return arr
            if len(kpts) > 0:
                m = cv2.KeyPoint_convert(list(kpts)).astype(float)
                return np.hstack((m, np.ones_like(m[..., 0, np.newaxis])))
            return np.empty((0, 3))
        self.m_top, self.m_bot = homo(self.kpts_top, m_top_array), homo(self.kpts_bot, m_bot_array)
        l = max(len(self.kpts_top), len(self.kpts_bot))
        if random_colors_RGB_list is None or len(random_colors_RGB_list) < l:
            self.random_colors_RGB = np.random.randint(low=0, high=256, size=(l, 3), dtype="uint8")
        else:
            self.random_colors_RGB = random_colors_RGB_list


# ---------------------------------------------------------------------------------------------------------------------
# Mono omnidirectional model (camera_models.py:862-2276, hot-path methods only)
# ---------------------------------------------------------------------------------------------------------------------
class OmniCamModel(object):
    def _init_default_values(self, **kwargs):
        self.F = np.array([0.0, 0.0, 0.0, 1.0]).reshape(4, 1)   # focus in [C], homogeneous column (camera_models.py:901)
        self.T_model_wrt_C = np.identity(4)
        self.T_C_wrt_model = np.identity(4)
        self.outer_img_radius = 0
        self.inner_img_radius = 0
        self.lowest_elevation_angle = -np.pi / 2
        self.highest_elevation_angle = np.pi / 2
        self.globally_lowest_elevation_angle = -np.pi / 2
        self.globally_highest_elevation_angle = np.pi / 2
        self.current_omni_img = None
        self.panorama = None
        self.mask = None
        self.units = "m"

    def set_pose(self, translation, rotation_matrix):
        """camera_models.py:955-962."""
        translation = np.asarray(translation, float)
        rotation_matrix = np.asarray(rotation_matrix, float)
        self.F[:3, 0] = translation[:3]
        self.T_model_wrt_C[:3, 3] = translation[:3]
        self.T_model_wrt_C[:3, :3] = rotation_matrix[:3, :3]
        self.T_C_wrt_model = np.identity(4)
        self.T_C_wrt_model[:3, :3] = rotation_matrix.T
        self.T_C_wrt_model[:3, 3] = -(rotation_matrix.T).dot(translation[:3])

    def map_angles_to_unit_sphere(self, theta, psi):
        """F8 (camera_models.py:1031-1065): homogeneous point(s) on the unit sphere for elevation theta, azimuth psi."""
        theta = np.asarray(theta, np.float64)
        psi = np.asarray(psi, np.float64)
        shape = np.broadcast(theta, psi).shape
        el = np.ascontiguousarray(np.broadcast_to(theta, shape).reshape(-1))
        az = np.ascontiguousarray(np.broadcast_to(psi, shape).reshape(-1))
        b = device_context().angles_to_sphere_f64(to_device(az), to_device(el)).cpu().numpy()
        # np.dstack((x, y, z, w)) of the reference: 0-D/1-D inputs come back as 1 x N x 4, 2-D inputs as rows x cols x 4
        out_shape = shape if len(shape) >= 2 else (1, int(np.prod(shape)) if len(shape) else 1)
        out = np.ones(out_shape + (4,))
        out[..., :3] = b.reshape(out_shape + (3,))
        return out

    def detect_sparse_features_on_panorama(self, feature_detection_method="ORB", num_of_features=50, median_win_size=0,
                                           show=True):
        """Per-bucket keypoints + ORB descriptors on the panorama (camera_models.py:1610-1797).  Returns (list of keypoint
        lists, list of N x 32 descriptor arrays), one entry per azimuthal mask.

        The reference's default detector, "GFT" (pose_est_tools.py:681), runs on the device (SURVEY §8f N3): 11 x 11 median
        blur of the BGR panorama, BGR2GRAY, goodFeaturesToTrack(maxCorners, 0.01, 5, mask) per mask, KeyPoint_convert,
        ORB.compute — sos_median_blur_11, sos_bgr_to_gray, sos_gft_detect, sos_orb_describe.  Other detectors stay on the
        host with OpenCV (they are not the reference's default path)."""
        pano = self.panorama.panoramic_img
        masks = self.panorama.azimuthal_masks or [None]
        if feature_detection_method.upper() == "GFT":
            if median_win_size not in (0, 11):
                raise NotImplementedError("the device median filter is 11 x 11 (the reference's median_win_size)")
            ctx = device_context()
            img = to_device(np.ascontiguousarray(pano))
            if pano.ndim == 3:
                if median_win_size > 0:
                    img = ctx.median_blur_11(img)
                gray = ctx.bgr_to_gray(img)
            else:
                gray = img          # camera_models.py:1712-1713: a single-channel panorama is used UNblurred (sic)
            key = tuple(id(m) for m in masks)
            if getattr(self, "_masks_key", None) != key:
                self._masks_dev = None if masks[0] is None else to_device(np.ascontiguousarray(np.stack(masks)))
                self._masks_key = key
            xy, cnt = ctx.gft_detect(gray, self._masks_dev, int(num_of_features), 0.01, 5.0)
            cnt = cnt.cpu().numpy()[0]
            pts = [xy[0, m, :int(cnt[m])] for m in range(len(masks))]
            allpts = torch.cat(pts) if len(pts) > 1 else pts[0]
            desc, keep = ctx.orb_describe(gray, allpts.contiguous())
            desc, keep, allxy = desc.cpu().numpy(), keep.cpu().numpy().astype(bool), allpts.cpu().numpy()
            kpts_list, desc_list, o = [], [], 0
            for m in range(len(masks)):
                sl = slice(o, o + int(cnt[m]))
                o += int(cnt[m])
                k = keep[sl]
                # cv2.KeyPoint_convert: size 1, angle -1, response 1, octave 0, class_id -1
                kpts_list.append([cv2.KeyPoint(float(x), float(y), 1.0, -1.0, 1.0, 0, -1) for x, y in allxy[sl][k]])
                desc_list.append(desc[sl][k])
            return kpts_list, desc_list
        gray = cv2.cvtColor(pano, cv2.COLOR_BGR2GRAY) if pano.ndim == 3 else pano
        if median_win_size > 0:
            gray = cv2.medianBlur(gray, median_win_size)
        orb = cv2.ORB_create(nfeatures=int(num_of_features))
        kpts_list, desc_list = [], []
        for mask in masks:
            k, d = orb.detectAndCompute(gray, mask)
            kpts_list.append(list(k))
            desc_list.append(d if d is not None else np.zeros((0, 32), np.uint8))
        return kpts_list, desc_list

    def get_direction_angles_from_pixel(self, m_omni):
        """camera_models.py:1183-1194."""
        return self.lift_pixel_to_unit_sphere_wrt_focus(m_omni, return_angles=True)[1:]

    def get_pixel_from_direction_angles(self, azimuth, elevation, visualize=False):
        Pw = self.get_3D_point_from_angles_wrt_focus(azimuth=azimuth, elevation=elevation)
        return self.get_pixel_from_3D_point_wrt_M(Pw)

    def set_omni_image(self, img, pano_width_in_pixels=1200, generate_panorama=False, idx=-1, view=True, apply_mask=True,
                       mask_RGB=None, fold_mask=None):
        """camera_models.py:1481-1503.  `fold_mask` (extension): remap the UNMASKED image with this mirror mask folded
        into the LUT — same pixels as masking first, without materialising the masked image."""
        from .panorama import Panorama
        self.current_omni_img = img
        if generate_panorama or self.panorama is None:
            self.panorama = Panorama(self, width=pano_width_in_pixels)
        bg = (0, 0, 0) if mask_RGB is None else (mask_RGB[2], mask_RGB[1], mask_RGB[0])
        self.panorama.set_panoramic_image(img, idx, view=False, mask=fold_mask, mask_BGR_color=bg)


# ---------------------------------------------------------------------------------------------------------------------
# Stereo (two-mirror) model (camera_models.py:2278-3499, hot-path methods only)
# ---------------------------------------------------------------------------------------------------------------------
class OmniStereoModel(object):
    def __init__(self, top_model, bottom_model, **kwargs):
        self.top_model = top_model
        self.bot_model = bottom_model
        self.units = top_model.units
        self.current_omni_img = None
        self.construct_new_mask = True
        self.mask_RGB_color = None
        self.T_Cest_wrt_Rgt = None
        self.feature_matcher_for_static_stereo = None
        self.feature_matcher_for_motion = None
        self.set_params(**kwargs)
        self.baseline = self.get_baseline()

    def set_params(self, **kwargs):
        """camera_models.py:2314-2387: radial bounds -> elevation limits, shared by both panoramas (:2795-2800)."""
        for name, model in (("top", self.top_model), ("bottom", self.bot_model)):
            for suffix in ("", "_inner", "_outer"):
                key = f"center_point_{name}{suffix}"
                c = kwargs.get(key, model.precalib_params.center_point)
                setattr(model.precalib_params, "center_point" + suffix, np.asarray(c, float))
        self.top_model.outer_img_radius = kwargs.get("radius_top_outer", self.top_model.outer_img_radius)
        self.top_model.inner_img_radius = kwargs.get("radius_top_inner", self.top_model.inner_img_radius)
        self.bot_model.outer_img_radius = kwargs.get("radius_bottom_outer", self.bot_model.outer_img_radius)
        self.bot_model.inner_img_radius = kwargs.get("radius_bottom_inner", self.bot_model.inner_img_radius)
        for m in (self.top_model, self.bot_model):
            if m.outer_img_radius > 0:
                m.set_elevation_limits_from_radii()
        hi = max(self.top_model.highest_elevation_angle, self.bot_model.highest_elevation_angle)
        lo = min(self.top_model.lowest_elevation_angle, self.bot_model.lowest_elevation_angle)
        for m in (self.top_model, self.bot_model):
            m.globally_highest_elevation_angle, m.globally_lowest_elevation_angle = hi, lo

    def get_baseline(self):
        return self.top_model.F[2, 0] - self.bot_model.F[2, 0]

    # ---- F2: masks (camera_models.py:2932-3025) ---------------------------------------------------------------------
    def _make_masks(self, shape):
        pt, pb = self.top_model.precalib_params, self.bot_model.precalib_params
        c = lambda p: tuple(int(v) for v in np.asarray(p).astype("int"))
        mask_top = np.zeros(shape, np.uint8)
        cv2.circle(mask_top, c(pt.center_point_outer), int(self.top_model.outer_img_radius), (255, 255, 255), -1, 8, 0)
        if self.top_model.inner_img_radius > 0:
            cv2.circle(mask_top, c(pt.center_point_inner), int(self.top_model.inner_img_radius), (0, 0, 0), -1, 8, 0)
            if self.bot_model.outer_img_radius > 0:
                cv2.circle(mask_top, c(pb.center_point_outer), int(self.bot_model.outer_img_radius), (0, 0, 0), -1, 8, 0)
        outer = np.zeros(shape, np.uint8)
        inner = np.zeros(shape, np.uint8)
        cv2.circle(outer, c(pb.center_point_outer), int(self.bot_model.outer_img_radius), (255, 255, 255), -1, 8, 0)
        cv2.circle(inner, c(pb.center_point_inner), int(self.top_model.inner_img_radius), (255, 255, 255), -1, 8, 0)
        mask_bot = cv2.bitwise_and(outer, inner)
        cv2.circle(mask_bot, c(pb.center_point_inner), int(self.bot_model.inner_img_radius), (0, 0, 0), -1, 8, 0)
        self.top_model.mask, self.bot_model.mask = mask_top, mask_bot
        self.construct_new_mask = False

    def get_fully_masked_images(self, omni_img=None, view=True, color_RGB=None):
        """Materialised masked images, for callers that want them (the frame path below never does)."""
        if omni_img is None:
            omni_img = self.current_omni_img
        if self.construct_new_mask or self.top_model.mask is None:
            self._make_masks(omni_img.shape[0:2])
        bg = np.zeros(3, np.uint8) if color_RGB is None else np.array([color_RGB[2], color_RGB[1], color_RGB[0]], np.uint8)
        out = []
        for m in (self.top_model.mask, self.bot_model.mask):
            img = np.empty_like(omni_img)
            img[...] = bg[: omni_img.shape[2]] if omni_img.ndim == 3 else bg[0]
            img[m != 0] = omni_img[m != 0]
            out.append(img)
        return out[0], out[1]

    def set_current_omni_image(self, img, pano_width_in_pixels=1200, generate_panoramas=False, idx=-1, view=False,
                               apply_mask=True, mask_RGB=None):
        """camera_models.py:3107-3120 — mask + both remaps in one fused kernel launch per view."""
        self.current_omni_img = img
        if apply_mask and (self.construct_new_mask or self.top_model.mask is None):
            self._make_masks(img.shape[0:2])
        for m in (self.top_model, self.bot_model):
            m.set_omni_image(img, pano_width_in_pixels=pano_width_in_pixels, generate_panorama=generate_panoramas, idx=idx,
                             view=False, apply_mask=False, mask_RGB=mask_RGB, fold_mask=m.mask if apply_mask else None)

    # ---- F5: stereo matching per azimuthal bucket (camera_models.py:3027-3101) --------------------------------------
    def match_features_panoramic_top_bottom(self, keypts_list_top, desc_list_top, keypts_list_bot, desc_list_bot,
                                            min_rectified_disparity=1, max_horizontal_diff=1, show_matches=False,
                                            win_name="Matches"):
        """All buckets in ONE segmented launch (query = bottom, train = top), sorted per bucket, gated by
        filter_pixel_correspondences; same return tuple as the reference."""
        kt, kb, dt, db, seg_q, seg_t = [], [], [], [], [0], [0]
        for top_k, top_d, bot_k, bot_d in zip(keypts_list_top, desc_list_top, keypts_list_bot, desc_list_bot):
            if len(top_k) == 0 or len(bot_k) == 0:
                continue
            kt += list(top_k); kb += list(bot_k)
            dt.append(np.asarray(top_d, np.uint8)); db.append(np.asarray(bot_d, np.uint8))
            seg_t.append(len(kt)); seg_q.append(len(kb))
        if not dt:
            raise ValueError("need at least one array to concatenate")  # what np.concatenate raises in the reference
        kt, kb = np.array(kt), np.array(kb)
        dt, db = np.concatenate(dt), np.concatenate(db)
        pt = cv2.KeyPoint_convert(list(kt)).astype(np.float32).reshape(-1, 2)
        pb = cv2.KeyPoint_convert(list(kb)).astype(np.float32).reshape(-1, 2)
        ctx = device_context()
        seg_q, seg_t = np.asarray(seg_q, np.int32), np.asarray(seg_t, np.int32)
        qs, ql, ts, tl = (to_device(a) for a in (seg_q[:-1], np.diff(seg_q), seg_t[:-1], np.diff(seg_t)))
        i0, d0, _, _ = ctx.hamming_top2(to_device(db), to_device(dt), qs, ql, ts, tl, int(np.diff(seg_q).max()),
                                        int(np.diff(seg_t).max()), want_second=False)
        oq, ot, od, oc = ctx.match_select(ops.MATCH_NN, i0, d0, None, qs, ql, ts, px_q=to_device(pb), px_t=to_device(pt),
                                          max_du=float(max_horizontal_diff), min_dv=float(min_rectified_disparity))
        oq, ot, oc = oq.cpu().numpy(), ot.cpu().numpy(), oc.cpu().numpy()
        rq = np.concatenate([oq[seg_q[s]:seg_q[s] + oc[s]] for s in range(len(oc))])
        rt = np.concatenate([ot[seg_q[s]:seg_q[s] + oc[s]] for s in range(len(oc))])
        m_top = np.hstack((pt[rt].astype(float), np.ones((len(rt), 1))))
        m_bot = np.hstack((pb[rq].astype(float), np.ones((len(rq), 1))))
        colors = np.random.randint(low=0, high=256, size=(len(rt), 3), dtype="uint8")
        return (m_top, kt[rt], dt[rt]), (m_bot, kb[rq], db[rq]), colors

    # ---- F10 / F11 (camera_models.py:3299-3364, 2420-2490) ------------------------------------------------------------
    def get_triangulated_point_from_direction_angles(self, dir_angs_top, dir_angs_bot, use_midpoint_triangulation=False):
        if not use_midpoint_triangulation:
            raise NotImplementedError("the SOS frame path uses the midpoint method (pose_est_tools.py:283,365)")
        az1, el1 = (np.asarray(a, np.float64) for a in dir_angs_top)
        az2, el2 = (np.asarray(a, np.float64) for a in dir_angs_bot)
        shape = az1.shape
        f = lambda a: to_device(np.ascontiguousarray(a.reshape(-1)))
        xyz, _ = device_context().triangulate_midpoint_f64(f(az1), f(el1), f(az2), f(el2), self.top_model.F[:3, 0],
                                                           self.bot_model.F[:3, 0])
        out = np.ones((1,) + (int(np.prod(shape)),) + (4,)) if len(shape) <= 1 else np.ones(shape + (4,))
        out[..., :3] = xyz.cpu().numpy().reshape(out.shape[:-1] + (3,))
        return out

    # ---- N4: dense triangulation of the panoramic disparity map (camera_models.py:2492-2538, 2567-2685) ----------------
    def triangulate_from_depth_map(self, min_disparity=1, max_disparity=0, roi_cols=None, use_midpoint_triangulation=True,
                                   **unused):
        """Point cloud of `self.disparity_map` (float32 rows x cols, linked to the top panorama).  Returns
        (points_3D_wrt_C_homo [1, N, 4], top_pano_points_coords [1, N, 2]) in the reference's order (u-major); colours
        and PCL export of generate_point_clouds (camera_models.py:2687-2790) are left to the caller."""
        if not use_midpoint_triangulation:
            raise NotImplementedError("only the midpoint method is implemented (see get_triangulated_point_from_direction_angles)")
        top, bot = self.top_model.panorama, self.bot_model.panorama
        disp = np.ascontiguousarray(self.disparity_map, np.float32)
        # Panorama.get_panorama_row_from_elevation(bot.lowest_elevation_angle) (panorama.py:676-689)
        lowest_row = float(np.uint((bot.cyl_height_max - np.tan(self.bot_model.lowest_elevation_angle)) / bot.pixel_size))
        xyz, valid = device_context().dense_triangulate(top.pano_vector(), bot.pano_vector(), to_device(disp),
                                                        self.top_model.F[:3, 0], self.bot_model.F[:3, 0],
                                                        float(min_disparity), float(max_disparity), lowest_row, roi_cols)
        vt = valid.cpu().numpy().astype(bool).T                       # [cols, rows]: u-major like np.indices(shape[::-1])
        pts = xyz.cpu().numpy().astype(np.float64).transpose(1, 0, 2)[vt]
        uu, vv = np.nonzero(vt)
        homo = np.ones((1, len(pts), 4))
        homo[0, :, :3] = pts
        return homo, np.stack([uu, vv], 1)[np.newaxis, ...]

    def filter_panoramic_points_due_to_range(self, xyz_points_wrt_C, min_3D_range=0, max_3D_range=0.):
        """camera_models.py:3299-3321: norm over the LAST axis of whatever is passed (the frame code passes N x 4)."""
        p = np.asarray(xyz_points_wrt_C, np.float64)
        shape = p.shape[:-1]
        if not (min_3D_range > 0 or max_3D_range > 0) or p.size == 0:
            return np.ones(shape, dtype=bool)
        flat = p.reshape(-1, p.shape[-1])
        homo = flat.shape[1] == 4 and np.all(flat[:, 3] == 1.0)
        if flat.shape[1] not in (3, 4) or (flat.shape[1] == 4 and not homo):
            raise ValueError("expected N x 3 points or N x 4 homogeneous points with w == 1")
        # re-use the triangulation kernel's range gate on the given points: feed it rays that meet at each point
        ctx = device_context()
        valid = ctx.range_gate(to_device(np.ascontiguousarray(flat[:, :3])), float(min_3D_range), float(max_3D_range), homo)
        return valid.cpu().numpy().astype(bool).reshape(shape)


# ---------------------------------------------------------------------------------------------------------------------
# F12: RGB-D camera model (camera_models.py:750-860)
# ---------------------------------------------------------------------------------------------------------------------
class RGBDCamModel(object):
    def __init__(self, **kwargs):
        self.fx = kwargs.get("fx", 525.0)
        self.fy = kwargs.get("fy", 525.0)
        self.center_x = kwargs.get("center_x", 319.5)
        self.center_y = kwargs.get("center_y", 239.5)
        self.focal_length_m = kwargs.get("focal_length_m", 1.0 / 1000.0)
        self.depth_is_Z = kwargs.get("depth_is_Z", True)
        self.units = kwargs.get("units", "m")
        self.scaling_factor = kwargs.get("scaling_factor", 1. / 1000.0)
        self.do_undistortion = kwargs.get("do_undistortion", False)
        self.K = np.array([[self.fx, 0, self.center_x], [0, self.fy, self.center_y], [0, 0, 1]])
        self.image_size = kwargs.get("image_size", None)
        self.T_model_wrt_C = np.identity(4)
        self.T_C_wrt_model = np.identity(4)
        self.T_Cest_wrt_Rgt = None
        self.feature_matcher_for_motion = None

    def cam_vector(self):
        return np.array([self.fx, self.fy, self.center_x, self.center_y, self.focal_length_m, float(bool(self.depth_is_Z))])

    def get_depth_Z(self, depth, uv_coords=None, verbose=False):
        """camera_models.py:781-799: radial depth -> Z over the whole map (identity when depth_is_Z)."""
        if self.depth_is_Z:
            return depth
        d = np.ascontiguousarray(depth, np.float32)
        return device_context().rgbd_depth_to_z(self.cam_vector(), to_device(d)).cpu().numpy().astype(np.float64)

    def get_XYZ(self, depth, u_coords=None, v_coords=None):
        """camera_models.py:835-860: XYZ (1 x N x 3, NaN where the depth is 0) at the given integer pixels."""
        d = np.ascontiguousarray(depth, np.float32)
        if u_coords is None or v_coords is None:
            vv, uu = np.mgrid[:d.shape[0], :d.shape[1]]
            u_coords, v_coords, shape = uu, vv, d.shape
        else:
            shape = None
        u = np.ascontiguousarray(np.asarray(u_coords).ravel().astype(np.int32))
        v = np.ascontiguousarray(np.asarray(v_coords).ravel().astype(np.int32))
        xyz, _, _ = device_context().rgbd_backproject(self.cam_vector(), to_device(d), to_device(u), to_device(v))
        out = xyz.cpu().numpy().astype(np.float64)
        return out.reshape(shape + (3,)) if shape is not None else out[np.newaxis, ...]
