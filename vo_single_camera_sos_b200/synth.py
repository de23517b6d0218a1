"""Synthetic SOS rigs, scenes and ORB-like features (the datasets of the reference are not available offline).

Everything here is input generation in NumPy: a random GUMS parameter set (two GUM mirrors on a common axis), a textured
box scene rendered into omni images through the GUM lifting, landmarks projected into both cylindrical panoramas with
pixel noise, 256-bit descriptors with bit-flip noise, distractors and planted ties, and a smooth random trajectory.
Geometry conventions follow the reference: panorama column <-> azimuth and row <-> elevation as in
omnistereo/panorama.py:616-642, GUM projection as in omnistereo/gum.py:2512-2562.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

GUM_FIELDS = ("xi1", "xi2", "xi3", "k1", "k2", "k3", "gamma1", "gamma2", "alpha_c", "u_center", "v_center",
              "l1", "l2", "l3", "p1", "p2", "plane_k", "use_distortion")


@dataclass
class Rig:
    width: int
    height: int
    gum_top: dict
    gum_bot: dict
    f_top: np.ndarray          # focus of the top mirror in [C]
    f_bot: np.ndarray
    elev_top: tuple            # (lowest, highest) elevation seen by the top mirror [rad]
    elev_bot: tuple
    radii_top: tuple           # (inner, outer) image radius of the top annulus [px]
    radii_bot: tuple
    pano_cols: int
    pano: dict = field(default_factory=dict)   # shared panorama geometry (both mirrors use the global elevation span)

    def gum_vector(self, which: str) -> np.ndarray:
        g = self.gum_top if which == "top" else self.gum_bot
        return np.array([float(g[k]) for k in GUM_FIELDS], np.float64)

    def pano_vector(self) -> np.ndarray:
        p = self.pano
        return np.array([p["cols"], p["rows"], p["pixel_size"], p["cyl_height_max"], p["cyl_circumference"], p["cyl_radius"]],
                        np.float64)

    def mask(self, which: str) -> np.ndarray:
        """Annular mirror masks, as OmniStereoModel.get_fully_masked_images paints them (camera_models.py:2963-2988)."""
        g = self.gum_top if which == "top" else self.gum_bot
        r_in, r_out = self.radii_top if which == "top" else self.radii_bot
        yy, xx = np.mgrid[:self.height, :self.width]
        r = np.hypot(xx - g["u_center"], yy - g["v_center"])
        return ((r >= r_in) & (r <= r_out)).astype(np.uint8) * 255


def _gum_radius(gamma, xi3, theta):
    return gamma * np.cos(theta) / np.abs(np.sin(theta) - xi3)


def make_rig(width: int, height: int, pano_cols: int, seed: int = 0) -> Rig:
    """Random GUMS parameter set in the ranges of SURVEY §8d, arranged so that the two mirrors share a vertical FOV."""
    rng = np.random.default_rng(seed)
    H = float(min(width, height))
    c = np.array([width / 2.0 - 0.5, height / 2.0 - 0.5]) + rng.uniform(-3, 3, 2)
    xi3 = rng.uniform(0.85, 0.95)
    elev_top = (np.deg2rad(-48.0), np.deg2rad(15.0))
    elev_bot = (np.deg2rad(-15.0), np.deg2rad(48.0))
    # top mirror fills the outer annulus (r grows with elevation), bottom mirror the inner one (r shrinks with elevation)
    r_top_out = 0.47 * H
    gamma_top = r_top_out / (np.cos(elev_top[1]) / (xi3 - np.sin(elev_top[1])))
    r_top_in = _gum_radius(gamma_top, xi3, elev_top[0])
    r_bot_out = 0.93 * r_top_in
    gamma_bot = r_bot_out / (np.cos(elev_bot[0]) / (np.sin(elev_bot[0]) + xi3))
    r_bot_in = _gum_radius(gamma_bot, -xi3, elev_bot[1])

    def gum(gamma, z_axis):
        d = dict(xi1=rng.uniform(-0.002, 0.002), xi2=rng.uniform(-0.002, 0.002), xi3=z_axis * xi3,
                 k1=rng.uniform(-0.004, 0.004), k2=rng.uniform(-0.0004, 0.0004), k3=0.0,
                 gamma1=gamma, gamma2=gamma * rng.uniform(0.998, 1.002), alpha_c=0.0, u_center=c[0], v_center=c[1],
                 l1=0.0, l2=0.0, l3=0.0, p1=0.0, p2=0.0, use_distortion=1.0)
        d["plane_k"] = d["xi3"] - z_axis  # gum.py:379-382
        return d

    baseline = rng.uniform(0.10, 0.15)
    rig = Rig(width, height, gum(gamma_top, 1.0), gum(gamma_bot, -1.0), np.array([0.0, 0.0, baseline]), np.zeros(3),
              elev_top, elev_bot, (r_top_in, r_top_out), (r_bot_in, r_bot_out), pano_cols)
    hi = max(elev_top[1], elev_bot[1])
    lo = min(elev_top[0], elev_bot[0])
    h_max, h_min = np.tan(hi), np.tan(lo)
    ps = 2 * np.pi / pano_cols
    rig.pano = dict(cols=pano_cols, rows=int(np.ceil((h_max - h_min) / ps)), pixel_size=ps, cyl_height_max=h_max,
                    cyl_height_min=h_min, cyl_circumference=2 * np.pi, cyl_radius=1.0)
    return rig


# ---------------------------------------------------------------------------------------------------------------
# Scene, trajectory, features
# ---------------------------------------------------------------------------------------------------------------
@dataclass
class Scene:
    half_extent: np.ndarray     # axis-aligned room [-hx,hx] x [-hy,hy] x [-hz,hz] in the world frame
    texture: np.ndarray         # [6, T, T, 3] uint8, one blocky-noise texture per wall
    landmarks: np.ndarray       # [L, 3] world points on the walls and on boxes inside the room
    descriptors: np.ndarray     # [L, 32] uint8


def make_scene(n_landmarks: int, seed: int = 0, tex: int = 64) -> Scene:
    rng = np.random.default_rng(seed + 1000)
    half = np.array([rng.uniform(3.0, 4.5), rng.uniform(3.0, 4.5), rng.uniform(1.8, 2.6)])
    texture = rng.integers(0, 256, (6, tex, tex, 3), dtype=np.uint8)
    # landmarks: 60 % on the walls, 40 % floating inside (boxes / furniture), all within 0.6 .. 6.5 m of the origin
    n_wall = int(0.6 * n_landmarks)
    pts = []
    while sum(len(p) for p in pts) < n_wall:
        d = rng.normal(size=(n_wall, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        t = np.min(half / np.abs(d), axis=1)
        pts.append(d * t[:, None])
    walls = np.concatenate(pts)[:n_wall]
    d = rng.normal(size=(n_landmarks - n_wall, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    inside = d * rng.uniform(0.6, 2.8, (len(d), 1))
    inside = np.clip(inside, -0.95 * half, 0.95 * half)
    land = np.concatenate([walls, inside])
    desc = rng.integers(0, 256, (n_landmarks, 32), dtype=np.uint8)
    return Scene(half, texture, land, desc)


def make_trajectory(n_frames: int, seed: int = 0):
    """Smooth random motion: |t| in [1,5] cm and rotation <= 3 deg per frame (SURVEY §8d). Returns T_C_wrt_W [n,4,4]."""
    rng = np.random.default_rng(seed + 2000)
    T = np.eye(4)
    out = [T.copy()]
    vel = rng.normal(size=3)
    axis = rng.normal(size=3)
    for _ in range(n_frames - 1):
        vel = 0.9 * vel + 0.1 * rng.normal(size=3)
        axis = 0.9 * axis + 0.1 * rng.normal(size=3)
        t = vel / np.linalg.norm(vel) * rng.uniform(0.01, 0.05)
        t[2] *= 0.2
        a = axis / np.linalg.norm(axis)
        ang = np.deg2rad(rng.uniform(0.2, 3.0))
        K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
        R = np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K
        step = np.eye(4)
        step[:3, :3], step[:3, 3] = R, t
        T = T @ step
        out.append(T.copy())
    return np.array(out)


def project_to_pano(rig: Rig, which: str, P_c: np.ndarray):
    """Points in [C] -> panorama pixel (u, v) of one mirror and visibility (inside that mirror's elevation band).
    Inverse of panorama.py:616-642: az = 2 pi - ps * u, el = atan2(h_max - ps * v, 1)."""
    f = rig.f_top if which == "top" else rig.f_bot
    lo, hi = rig.elev_top if which == "top" else rig.elev_bot
    d = P_c - f
    az = np.mod(np.arctan2(d[:, 1], d[:, 0]), 2 * np.pi)
    az = np.where(az == 0, 2 * np.pi, az)
    el = np.arctan2(d[:, 2], np.hypot(d[:, 0], d[:, 1]))
    p = rig.pano
    u = (p["cyl_circumference"] - az) / p["pixel_size"]
    v = (p["cyl_height_max"] - np.tan(el)) / p["pixel_size"]
    vis = (el >= lo) & (el <= hi) & (u >= 0) & (u < p["cols"]) & (v >= 0) & (v < p["rows"])
    return np.stack([u, v], 1), vis, az


def make_frame_features(rig: Rig, scene: Scene, T_c_wrt_w: np.ndarray, n_per_view: int, n_buckets: int, seed: int,
                        cap: int, flip: float = 0.08, px_sigma: float = 0.15, distractors: float = 0.25, n_ties: int = 8,
                        dynamic: float = 0.0):
    """Features of one frame for both views, bucketed by azimuth (30 deg buckets, pose_est_tools.py:871-878).

    dynamic: fraction of the landmarks that MOVE between frames (a fixed subset, chosen by landmark id): in every frame
    each of them is displaced by an own random rotation of 8..20 degrees about the camera centre.  They still match by
    descriptor (stereo and temporal) and triangulate consistently within a frame, but their temporal correspondences
    violate the rigid motion by more than the 5 degree RANSAC threshold: outliers.  dynamic = 0.65 gives the 35 % inlier
    rate the reference assumes (outlier fraction 0.65, pose_est_tools.py:675; SURVEY 8d).

    Returns per view: px [cap,2] float32, desc [cap,32] uint8, bucket_off [n_buckets+1] int32, landmark id [cap] (-1 for
    distractors); rows beyond bucket_off[-1] are padding."""
    rng = np.random.default_rng(seed)
    Tw2c = np.linalg.inv(T_c_wrt_w)
    P_c = scene.landmarks @ Tw2c[:3, :3].T + Tw2c[:3, 3]
    if dynamic > 0.0:
        L = len(P_c)
        dyn = ((np.arange(L, dtype=np.uint64) * np.uint64(2654435761)) % np.uint64(1000)) < np.uint64(int(round(dynamic * 1000)))
        rd = np.random.default_rng(seed + 99991)          # own stream: the static features are those of dynamic = 0
        ax = rd.normal(size=(L, 3))
        ax /= np.linalg.norm(ax, axis=1, keepdims=True)
        ang = np.deg2rad(rd.uniform(8.0, 20.0, L))[:, None]
        # Rodrigues: p cos(a) + (k x p) sin(a) + k (k.p) (1 - cos(a))
        rot = P_c * np.cos(ang) + np.cross(ax, P_c) * np.sin(ang) + ax * np.sum(ax * P_c, axis=1, keepdims=True) * (1 - np.cos(ang))
        P_c = np.where(dyn[:, None], rot, P_c)
    out = {}
    # both views favour landmarks visible in both mirrors so that stereo matching has something to find
    vis_both = None
    proj = {}
    for which in ("top", "bot"):
        uv, vis, az = project_to_pano(rig, which, P_c)
        rngd = np.linalg.norm(P_c, axis=1)
        vis &= (rngd > 0.45) & (rngd < 8.0)
        proj[which] = (uv, vis, az)
        vis_both = vis if vis_both is None else (vis_both & vis)
    common = np.nonzero(vis_both)[0]
    for which in ("top", "bot"):
        uv, vis, az = proj[which]
        n_true = int(round(n_per_view * (1.0 - distractors)))
        only = np.nonzero(vis & ~vis_both)[0]
        n_common = min(len(common), int(0.85 * n_true))
        ids = np.concatenate([rng.permutation(common)[:n_common], rng.permutation(only)[: n_true - n_common]])
        px = uv[ids] + rng.normal(0, px_sigma, (len(ids), 2))
        desc = scene.descriptors[ids] ^ np.packbits(rng.random((len(ids), 256)) < flip, axis=1)
        n_dis = n_per_view - len(ids)
        p = rig.pano
        lo, hi = rig.elev_top if which == "top" else rig.elev_bot
        v_lo = (p["cyl_height_max"] - np.tan(hi)) / p["pixel_size"]
        v_hi = (p["cyl_height_max"] - np.tan(lo)) / p["pixel_size"]
        px_d = np.stack([rng.uniform(0, p["cols"], n_dis), rng.uniform(v_lo, min(v_hi, p["rows"] - 1e-3), n_dis)], 1)
        desc_d = rng.integers(0, 256, (n_dis, 32), dtype=np.uint8)
        px = np.concatenate([px, px_d])
        desc = np.concatenate([desc, desc_d])
        lid = np.concatenate([ids, np.full(n_dis, -1)])
        px[:, 0] = np.clip(px[:, 0], 0, p["cols"] - 1e-3)
        px[:, 1] = np.clip(px[:, 1], 0, p["rows"] - 1e-3)
        # planted exact descriptor ties (lowest index must win)
        for _ in range(n_ties):
            a, b = rng.integers(0, len(px), 2)
            desc[b] = desc[a]
        # bucket by azimuth: az = 2 pi - ps u, bucket k covers [k, k+1) * (2 pi / n_buckets)
        azp = p["cyl_circumference"] - p["pixel_size"] * px[:, 0].astype(np.float32).astype(np.float64)
        bucket = np.clip((azp / (2 * np.pi / n_buckets)).astype(int), 0, n_buckets - 1)
        order = np.argsort(bucket, kind="stable")
        px, desc, lid, bucket = px[order], desc[order], lid[order], bucket[order]
        off = np.concatenate([[0], np.cumsum(np.bincount(bucket, minlength=n_buckets))]).astype(np.int32)
        pxo = np.zeros((cap, 2), np.float32)
        deo = np.zeros((cap, 32), np.uint8)
        lio = np.full(cap, -2, np.int64)
        n = len(px)
        pxo[:n], deo[:n], lio[:n] = px.astype(np.float32), desc, lid
        out[which] = dict(px=pxo, desc=deo, bucket_off=off, landmark=lio)
    return out


def render_omni(rig: Rig, scene: Scene, T_c_wrt_w: np.ndarray, lift=None) -> np.ndarray:
    """Omni image [H,W,3] uint8: every pixel inside a mirror annulus is lifted to its viewing ray (GUM lifting,
    gum.py:2673-2762), the ray is cast from that mirror's focus into the textured room and the wall texture is sampled
    (nearest, blocky cells).  `lift(which, uv[n,2]) -> sphere[n,3]` lets the caller run the lifting on the device."""
    from . import _synth_lift
    H, W = rig.height, rig.width
    img = np.zeros((H, W, 3), np.uint8)
    yy, xx = np.mgrid[:H, :W]
    R, t = T_c_wrt_w[:3, :3], T_c_wrt_w[:3, 3]
    for which in ("top", "bot"):
        m = rig.mask(which) != 0
        uv = np.stack([xx[m], yy[m]], 1).astype(np.float64)
        g = rig.gum_top if which == "top" else rig.gum_bot
        d_c = lift(which, uv) if lift is not None else _synth_lift.gum_lift(g, uv)
        f = rig.f_top if which == "top" else rig.f_bot
        o = R @ f + t
        d = d_c @ R.T
        with np.errstate(divide="ignore", invalid="ignore"):
            tt = np.where(d > 0, (scene.half_extent - o) / d, (-scene.half_extent - o) / d)
        k = np.argmin(tt, axis=1)
        hit = o + d * np.min(tt, axis=1, keepdims=True)
        face = 2 * k + (d[np.arange(len(d)), k] > 0)
        a = (k + 1) % 3
        b = (k + 2) % 3
        T = scene.texture.shape[1]
        cell = 0.12  # metres per texture cell
        iu = np.mod(np.floor(hit[np.arange(len(d)), a] / cell).astype(int), T)
        iv = np.mod(np.floor(hit[np.arange(len(d)), b] / cell).astype(int), T)
        img[m] = scene.texture[face, iu, iv]
    return img


# ---------------------------------------------------------------------------------------------------------------
# RGB-D sequences (BASELINE configuration 5, demo_vo_rgbd.py)
# ---------------------------------------------------------------------------------------------------------------
RGBD_FIELDS = ("fx", "fy", "center_x", "center_y", "focal_length_m", "depth_is_Z")


@dataclass
class RgbdSequence:
    cam: dict                  # RGBD_FIELDS -> value (RGBDCamModel's intrinsics, camera_models.py:752-779)
    trajectory: np.ndarray     # T_C_wrt_W [n, 4, 4]
    landmarks: np.ndarray      # [L, 3] world points
    frames: list               # per frame: depth [480, 640] float32, px [n, 2] float32, desc [n, 32] uint8, landmark [n]
                               # int64 (-1 = distractor)
    background: float = 0.0

    def cam_vector(self) -> np.ndarray:
        return np.array([float(self.cam[k]) for k in RGBD_FIELDS], np.float64)

    def inputs(self, ids, max_kp: int) -> dict:
        """The frames `ids` as the RGB-D front-end's step inputs: depth [B,h,w] f32, px [B,max_kp,2] f32, desc
        [B,max_kp,32] u8 (rows past a frame's keypoints are zero), n_kp [B] int32."""
        fr = [self.frames[i] for i in ids]
        h, w = fr[0]["depth"].shape
        out = dict(depth=np.stack([f["depth"] for f in fr]), px=np.zeros((len(fr), max_kp, 2), np.float32),
                   desc=np.zeros((len(fr), max_kp, 32), np.uint8), n_kp=np.zeros(len(fr), np.int32))
        for b, f in enumerate(fr):
            n = min(len(f["px"]), max_kp)
            out["px"][b, :n], out["desc"][b, :n], out["n_kp"][b] = f["px"][:n], f["desc"][:n], n
        return out


def rgbd_depth_value(cam: dict, Z: np.ndarray, u: np.ndarray, v: np.ndarray) -> np.ndarray:
    """What the sensor stores at integer pixel (u, v) for a point at depth Z: Z itself, or for radial maps the distance
    along the pixel's ray, the inverse of RGBDCamModel.get_depth_Z (camera_models.py:781-799)."""
    if cam["depth_is_Z"]:
        return np.asarray(Z, np.float64)
    ray = np.sqrt(((u - cam["center_x"]) / cam["fx"]) ** 2 + ((v - cam["center_y"]) / cam["fy"]) ** 2 + 1.0)
    return Z * ray


def make_rgbd_sequence(n_frames: int, n_kp: int = 2000, depth_is_Z: bool = True, seed: int = 0, flip: float = 0.04,
                       distractors: float = 0.25, width: int = 640, height: int = 480,
                       background: float = 0.0) -> RgbdSequence:
    """A pinhole RGB-D camera moving along make_trajectory through a room of landmarks (walls, and points floating inside
    at 0.7 .. 3 m), intrinsics of demo_vo_rgbd.py: fx = fy = 525 for Z depth maps, 554.256258 for radial ones (the
    synthetic branch), c = (319.5, 239.5).

    Per frame, n_kp keypoints in random order: about (1 - distractors) of them are landmarks in view (pixel = the float32
    projection, descriptor = the landmark's with per-view bit flips of probability `flip`), the rest distractors (uniform
    pixel, random descriptor); the landmarks chosen are the strongest in view by a fixed per-landmark strength, so that
    consecutive frames share most of them.  The depth map is `background` everywhere except at the truncated pixel of every
    landmark keypoint, which holds that landmark's depth; of two landmarks that truncate to the same pixel the nearer
    one (then the lower id) is kept and the other is not a keypoint.  The default background 0 is "no reading": a keypoint
    there has no 3D point (camera_models.py:846), so distractors mostly drop out at the range gate and the temporal
    correspondences are nearly outlier-free (one outlier inside the 5 degree RANSAC threshold already pulls the LM pose
    of the reference's bearing residual away from the true motion)."""
    cam = dict(fx=525.0 if depth_is_Z else 554.256258, fy=525.0 if depth_is_Z else 554.256258, center_x=319.5,
               center_y=239.5, focal_length_m=1.0 / 1000.0, depth_is_Z=1.0 if depth_is_Z else 0.0)
    rng = np.random.default_rng(seed + 3000)
    half = np.array([4.0, 4.0, 2.5])
    n_land = max(24 * n_kp, 2000)
    d = rng.normal(size=(n_land, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    walls = d * np.min(half / np.abs(d), axis=1, keepdims=True)
    inside = d * rng.uniform(0.7, 3.0, (n_land, 1))
    land = np.where((np.arange(n_land) % 5 < 3)[:, None], walls, inside)   # 60 % walls, 40 % inside
    land_desc = rng.integers(0, 256, (n_land, 32), dtype=np.uint8)
    strength = rng.random(n_land)      # a detector finds the same strong corners again from frame to frame
    traj = make_trajectory(n_frames, seed)
    n_true = int(round(n_kp * (1.0 - distractors)))
    frames = []
    for fi, T in enumerate(traj):
        fr = np.random.default_rng([seed, fi, 17])
        P = (land - T[:3, 3]) @ T[:3, :3]                     # R^T (p - t): world -> camera
        Z = P[:, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            uv = np.stack([cam["fx"] * P[:, 0] / Z + cam["center_x"], cam["fy"] * P[:, 1] / Z + cam["center_y"]], 1)
        uv32 = uv.astype(np.float32)
        tu, tv = np.trunc(uv32[:, 0]), np.trunc(uv32[:, 1])
        vis = (Z > 0.5) & (tu >= 0) & (tu < width) & (tv >= 0) & (tv < height)
        vis_ids = np.flatnonzero(vis)
        ids = vis_ids[np.argsort(-strength[vis_ids], kind="stable")[:n_true]]   # the strongest corners in view
        # one landmark per truncated pixel: nearest first, then lowest id
        pix = tv[ids].astype(np.int64) * width + tu[ids].astype(np.int64)
        order = np.lexsort((ids, Z[ids]))
        _, first = np.unique(pix[order], return_index=True)
        ids = ids[np.sort(order[first])]
        ui, vi = tu[ids].astype(np.int64), tv[ids].astype(np.int64)
        depth = np.full((height, width), background, np.float32)
        depth[vi, ui] = rgbd_depth_value(cam, Z[ids], ui, vi).astype(np.float32)
        n_dis = n_kp - len(ids)
        px = np.concatenate([uv32[ids], np.stack([fr.uniform(0, width, n_dis), fr.uniform(0, height, n_dis)], 1)])
        px = px.astype(np.float32)
        desc = np.concatenate([land_desc[ids] ^ np.packbits(fr.random((len(ids), 256)) < flip, axis=1),
                               fr.integers(0, 256, (n_dis, 32), dtype=np.uint8)])
        lid = np.concatenate([ids, np.full(n_dis, -1)]).astype(np.int64)
        perm = fr.permutation(n_kp)
        frames.append(dict(depth=depth, px=px[perm], desc=desc[perm], landmark=lid[perm]))
    return RgbdSequence(cam, traj, land, frames, background)
