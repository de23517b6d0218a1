"""Python handle on the batched GPU-resident SOS front-end (sos_frontend_* in include/sosfront.h).

`Frontend.step(...)` takes device tensors, `Frontend.step_host(...)` / `submit_host` + `wait_host` take pinned host
arrays (the end-to-end path: H2D, kernels, D2H).  After `set_detector(...)`, `step_images` / `step_host_images` take the
omni images alone and detect the features inside the step.  A `Frontend` made from an `RgbdFrontendConfig` is the RGB-D
front-end (BASELINE configuration 5): `step_rgbd` / `step_host_rgbd` take depth maps and keypoints.  All data-dependent
sizes stay on the device; see csrc/frontend.cu.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np
import torch

from . import ops
from ._lib import check


class _Config(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("src_h", C.c_int32), ("src_w", C.c_int32), ("channels", C.c_int32),
        ("pano_rows", C.c_int32), ("pano_cols", C.c_int32), ("n_buckets", C.c_int32),
        ("max_feat_per_view", C.c_int32), ("max_feat_per_bucket", C.c_int32), ("cap", C.c_int32),
        ("n_hyp", C.c_int32), ("score_mode", C.c_int32), ("homogeneous_norm", C.c_int32), ("refit", C.c_int32),
        ("refine_iters", C.c_int32), ("keyframe_mode", C.c_int32), ("solver", C.c_int32),
        ("ransac_threshold", C.c_double), ("stereo_max_du", C.c_double), ("stereo_min_dv", C.c_double),
        ("temporal_max_du", C.c_double), ("min_range", C.c_double), ("max_range", C.c_double),
        ("pano_top", C.c_double * 6), ("pano_bot", C.c_double * 6), ("f_top", C.c_double * 3), ("f_bot", C.c_double * 3),
        ("rig", C.c_double * 24), ("border", C.c_uint8 * 4), ("background", C.c_uint8 * 4),
    ]


_BUF_FIELDS = [
    ("pano", "u8"), ("st_q_start", "i32"), ("st_q_len", "i32"), ("st_t_start", "i32"), ("st_t_len", "i32"),
    ("st_idx0", "i32"), ("st_d0", "i32"), ("st_pair_q", "i32"), ("st_pair_t", "i32"), ("st_pair_d", "i32"),
    ("st_pair_count", "i32"), ("uv_c", "f32"), ("uv_top", "f32"), ("uv_bot", "f32"), ("b_top", "f32"), ("b_bot", "f32"),
    ("xyz", "f32"), ("src_top", "i32"), ("src_bot", "i32"), ("n", "i32"), ("desc_c", "i32"),
    ("tm_q_start", "i32"), ("tm_q_len", "i32"), ("tm_t_start", "i32"), ("tm_t_len", "i32"),
    ("tm_idx0", "i32"), ("tm_d0", "i32"), ("tm_pair_q", "i32"), ("tm_pair_t", "i32"), ("tm_pair_d", "i32"),
    ("tm_pair_count", "i32"), ("p_ref", "f32"), ("p_cur", "f32"), ("f_cur", "f32"), ("cam", "u8"),
    ("n_corr", "i32"), ("n_corr_top", "i32"), ("ransac_pose", "f32"), ("pose", "f32"), ("best_hyp", "i32"),
    ("best_count", "i32"), ("n_refit", "i32"), ("inlier_mask", "u8"), ("stats", "i32"), ("refine_stats", "f64"), ("ref_slot", "i32"),
    ("overflow", "i32"),
]


class _Buffers(C.Structure):
    _fields_ = [(name, C.c_void_p) for name, _ in _BUF_FIELDS] + [
        ("batch", C.c_int32), ("cap", C.c_int32), ("launches_per_step", C.c_int32), ("views", C.c_int32)]


class _RgbdConfig(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("max_kp", C.c_int32), ("n_hyp", C.c_int32),
        ("solver", C.c_int32), ("refit", C.c_int32), ("refine_iters", C.c_int32), ("keyframe_mode", C.c_int32),
        ("cam", C.c_double * len(ops.RGBD_FIELDS)), ("min_z", C.c_double), ("max_z", C.c_double),
        ("temporal_max_du", C.c_double), ("ransac_threshold", C.c_double),
    ]


@dataclass
class RgbdFrontendConfig:
    """The RGB-D front-end (sos_rgbd_frontend_config); defaults follow RGBDFrame / TrackerRGBDSE3
    (pose_est_tools.py:429-430, 672-707, 880-958)."""
    batch: int
    cam: Sequence[float]               # ops.RGBD_FIELDS order: fx, fy, center_x, center_y, focal_length_m, depth_is_Z
    height: int = 480
    width: int = 640
    max_kp: int = 2000                 # keypoint rows per frame, and the store capacity
    n_hyp: int = 210
    solver: int = 0                    # ops.SOLVER_ARUN (hyp [n_hyp,3]) / ops.SOLVER_P3P (hyp [n_hyp,4])
    refit: int = 2                     # ops.REFINE_LM: the tracker's absolute_pose_optimize_nonlinear
    refine_iters: int = 0              # REFINE_LM: maximum cost evaluations (0 -> 20)
    keyframe_mode: bool = False
    min_z: float = 0.8
    max_z: float = 7.0
    temporal_max_du: Optional[float] = None    # None -> 0.5 * 2 * center_x (pose_est_tools.py:958)
    ransac_threshold: float = 1.0 - math.cos(math.radians(5.0))

    def to_c(self) -> _RgbdConfig:
        c = _RgbdConfig()
        for k in ("batch", "height", "width", "max_kp", "n_hyp", "solver", "refit", "refine_iters"):
            setattr(c, k, int(getattr(self, k)))
        c.keyframe_mode = int(bool(self.keyframe_mode))
        cam = [float(x) for x in self.cam]
        if len(cam) != len(ops.RGBD_FIELDS):
            raise ValueError(f"cam must hold {len(ops.RGBD_FIELDS)} values ({', '.join(ops.RGBD_FIELDS)})")
        c.cam[:] = cam
        c.min_z, c.max_z = float(self.min_z), float(self.max_z)
        c.temporal_max_du = float(0.5 * 2.0 * cam[2] if self.temporal_max_du is None else self.temporal_max_du)
        c.ransac_threshold = float(self.ransac_threshold)
        return c


@dataclass
class FrontendConfig:
    """Defaults follow the reference (pose_est_tools.py:284-308, 672-707, 862-878)."""
    batch: int
    src_h: int
    src_w: int
    pano_rows: int
    pano_cols: int
    pano_top: Sequence[float]          # ops.PANO_FIELDS order
    pano_bot: Sequence[float]
    f_top: Sequence[float]             # mirror foci in [C]
    f_bot: Sequence[float]
    channels: int = 3
    n_buckets: int = 12
    max_feat_per_view: int = 8192
    max_feat_per_bucket: int = 1024
    cap: int = 8192
    n_hyp: int = 210
    score_mode: int = ops.SCORE_BEARING
    ransac_threshold: float = 1.0 - math.cos(math.radians(5.0))
    homogeneous_norm: bool = True
    refit: int = 1                    # ops.REFINE_NONE / REFINE_ARUN / REFINE_LM (True == REFINE_ARUN)
    refine_iters: int = 0             # REFINE_LM: maximum cost evaluations (0 -> 20)
    keyframe_mode: bool = False       # track against reference slots (set_ref_slots / promote / retrack)
    solver: int = 0                   # ops.SOLVER_ARUN (hyp [n_hyp,3]) / ops.SOLVER_P3P (bearing-only, hyp [n_hyp,4])
    stereo_max_du: float = 2.5
    stereo_min_dv: float = 1.0
    temporal_max_du: Optional[float] = None   # None -> 0.125 * 0.5 * pano_cols
    min_range: float = 0.5
    max_range: float = 7.0
    rig: Optional[Sequence[float]] = None      # 2 x [Rc|tc]; None -> identity rotations at the foci
    border: Sequence[int] = (0, 0, 0, 0)
    background: Sequence[int] = (0, 0, 0, 0)

    def to_c(self) -> _Config:
        c = _Config()
        for k in ("batch", "src_h", "src_w", "channels", "pano_rows", "pano_cols", "n_buckets", "max_feat_per_view",
                  "max_feat_per_bucket", "cap", "n_hyp", "score_mode"):
            setattr(c, k, int(getattr(self, k)))
        c.homogeneous_norm = int(bool(self.homogeneous_norm))
        c.refit = int(self.refit)
        c.refine_iters = int(self.refine_iters)
        c.keyframe_mode = int(bool(self.keyframe_mode))
        c.solver = int(self.solver)
        c.ransac_threshold = float(self.ransac_threshold)
        c.stereo_max_du, c.stereo_min_dv = float(self.stereo_max_du), float(self.stereo_min_dv)
        c.temporal_max_du = float(0.125 * 0.5 * self.pano_cols if self.temporal_max_du is None else self.temporal_max_du)
        c.min_range, c.max_range = float(self.min_range), float(self.max_range)
        c.pano_top[:] = [float(x) for x in self.pano_top]
        c.pano_bot[:] = [float(x) for x in self.pano_bot]
        c.f_top[:] = [float(x) for x in self.f_top]
        c.f_bot[:] = [float(x) for x in self.f_bot]
        rig = self.rig
        if rig is None:
            rig = np.zeros((2, 3, 4))
            rig[:, :, :3] = np.eye(3)
            rig[0, :, 3] = self.f_top
            rig[1, :, 3] = self.f_bot
        c.rig[:] = [float(x) for x in np.asarray(rig, np.float64).reshape(-1)]
        b = list(self.border) + [0] * 4
        g = list(self.background) + [0] * 4
        c.border[:] = [int(x) for x in b[:4]]
        c.background[:] = [int(x) for x in g[:4]]
        return c


class _DetectConfig(C.Structure):
    _fields_ = [("corners_per_bucket", C.c_int32), ("median", C.c_int32), ("quality_level", C.c_double),
                ("min_distance", C.c_double)]


_FEATURE_FIELDS = ["px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot", "detect_stats"]


class _Features(C.Structure):
    _fields_ = [(name, C.c_void_p) for name in _FEATURE_FIELDS]


class _DeviceArray:
    """Wraps a raw device pointer so torch can view it (no copy, no ownership)."""

    def __init__(self, ptr: int, shape, typestr: str, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 2}
        self._owner = owner


_TYPES = {"u8": ("|u1", torch.uint8), "i32": ("<i4", torch.int32), "f32": ("<f4", torch.float32),
          "f64": ("<f8", torch.float64)}


class Frontend:
    def __init__(self, ctx: ops.Context, cfg, lut: Optional[torch.Tensor], hyp: torch.Tensor):
        """SOS (cfg: FrontendConfig): lut [2, rows, cols] int64 (packed LUT of the top and bottom view).  RGB-D (cfg:
        RgbdFrontendConfig): lut is None.  hyp [n_hyp, 3] int32 (uint32 bits; [n_hyp, 4] for SOLVER_P3P)."""
        self.ctx, self.cfg = ctx, cfg
        self.rgbd = isinstance(cfg, RgbdFrontendConfig)
        ctx._sync_stream()
        if self.rgbd:
            if lut is not None:
                raise ValueError("the RGB-D front-end takes no LUT")
        elif tuple(lut.shape) != (2, cfg.pano_rows, cfg.pano_cols):
            raise ValueError("lut must be [2, pano_rows, pano_cols]")
        if hyp.shape[0] != cfg.n_hyp or hyp.shape[1] != (4 if cfg.solver == ops.SOLVER_P3P else 3):
            raise ValueError("hyp must be [n_hyp, 3] (SOLVER_ARUN) or [n_hyp, 4] (SOLVER_P3P)")
        self._lut, self._hyp = lut, hyp  # keep alive
        self._c = cfg.to_c()
        h = C.c_void_p()
        if self.rgbd:
            check(ctx.lib.sos_frontend_create_rgbd(ctx._h, C.byref(self._c), ctx._t(hyp, torch.int32, "hyp"), C.byref(h)))
        else:
            check(ctx.lib.sos_frontend_create(ctx._h, C.byref(self._c), ctx._t(lut, torch.int64, "lut"),
                                              ctx._t(hyp, torch.int32, "hyp"), C.byref(h)))
        self._h = h
        self._stream = torch.cuda.current_stream(ctx.device)

    def _need(self, rgbd: bool, what: str):
        if self.rgbd != rgbd:
            raise TypeError(f"{what} needs {'an RGB-D' if rgbd else 'an SOS'} front-end")

    def close(self):
        if getattr(self, "_h", None):
            self.ctx.lib.sos_frontend_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        check(self.ctx.lib.sos_frontend_reset(self._h))

    def set_graph(self, enabled: bool):
        check(self.ctx.lib.sos_frontend_set_graph(self._h, int(enabled)))

    def profile_begin(self):
        """Per-launch CUDA-event timing of the following steps (they run eagerly, not from the graph)."""
        check(self.ctx.lib.sos_frontend_profile_begin(self._h))

    def profile_end(self, max_n: int = 4096):
        """-> list of (entry point name, milliseconds) in launch order."""
        names = C.create_string_buffer(64 * max_n)
        ms = (C.c_float * max_n)()
        n = C.c_int()
        check(self.ctx.lib.sos_frontend_profile_end(self._h, names, len(names), ms, max_n, C.byref(n)))
        nm = names.value.decode().split("\n")[: n.value]
        return [(nm[i], float(ms[i])) for i in range(n.value)]

    def _check_inputs(self, omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot, on_device: bool):
        self._need(False, "step / submit_host")
        c = self.cfg
        shapes = {
            "omni": ((c.batch, c.src_h, c.src_w, c.channels), (torch.uint8, np.uint8)),
            "px_top": ((c.batch, c.max_feat_per_view, 2), (torch.float32, np.float32)),
            "px_bot": ((c.batch, c.max_feat_per_view, 2), (torch.float32, np.float32)),
            "desc_top": ((c.batch, c.max_feat_per_view, 32), (torch.uint8, np.uint8)),
            "desc_bot": ((c.batch, c.max_feat_per_view, 32), (torch.uint8, np.uint8)),
            "boff_top": ((c.batch, c.n_buckets + 1), (torch.int32, np.int32)),
            "boff_bot": ((c.batch, c.n_buckets + 1), (torch.int32, np.int32)),
        }
        vals = dict(omni=omni, px_top=px_top, desc_top=desc_top, boff_top=boff_top, px_bot=px_bot, desc_bot=desc_bot,
                    boff_bot=boff_bot)
        ptrs = {}
        for k, v in vals.items():
            shape, (tdt, ndt) = shapes[k]
            if tuple(v.shape) != shape:
                raise ValueError(f"{k}: expected shape {shape}, got {tuple(v.shape)}")
            if on_device:
                ptrs[k] = self.ctx._t(v, tdt, k)
            else:
                if isinstance(v, torch.Tensor):
                    if v.is_cuda or v.dtype != tdt or not v.is_contiguous():
                        raise TypeError(f"{k}: expected a contiguous host tensor of {tdt}")
                    ptrs[k] = v.data_ptr()
                else:
                    if v.dtype != ndt or not v.flags.c_contiguous:
                        raise TypeError(f"{k}: expected a C-contiguous host array of {ndt}")
                    ptrs[k] = v.ctypes.data
                if k.startswith("boff"):
                    # host path: the offsets are at hand, so refuse what the device path can only clamp and count
                    # (buffers()["overflow"]): non-monotonic offsets, rows beyond max_feat_per_view, oversized buckets
                    o = np.asarray(v)
                    w = np.diff(o, axis=1)
                    if o.min() < 0 or o.max() > c.max_feat_per_view or w.min() < 0:
                        raise ValueError(f"{k}: bucket offsets must be non-decreasing within [0, max_feat_per_view]")
                    if w.max() > c.max_feat_per_bucket:
                        raise ValueError(f"{k}: a bucket holds {int(w.max())} features, max_feat_per_bucket is "
                                         f"{c.max_feat_per_bucket}")
        return [ptrs[k] for k in ("omni", "px_top", "desc_top", "boff_top", "px_bot", "desc_bot", "boff_bot")]

    def step(self, omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot):
        """Asynchronous step on device tensors; results are read through `buffers()`."""
        p = self._check_inputs(omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot, True)
        self.ctx._sync_stream()   # fence against torch's CURRENT stream (the caller may have switched it since create)
        check(self.ctx.lib.sos_frontend_step(self._h, *p))

    def submit_host(self, omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot) -> int:
        p = self._check_inputs(omni, px_top, desc_top, boff_top, px_bot, desc_bot, boff_bot, False)
        t = C.c_int()
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_submit_host(self._h, *p, C.byref(t)))
        return t.value

    def wait_host(self, ticket: int):
        poses = np.empty((self.cfg.batch, 3, 4), np.float32)
        stats = np.empty((self.cfg.batch, 4), np.int32)
        check(self.ctx.lib.sos_frontend_wait_host(self._h, int(ticket), poses.ctypes.data, stats.ctypes.data))
        return poses, stats

    # -- keyframe mode (sos_frontend_config.keyframe_mode) ---------------------------------------------------------
    def set_ref_slots(self, slots: Sequence[int]):
        arr = np.ascontiguousarray(np.asarray(slots, np.int32))
        if arr.shape != (self.cfg.batch,):
            raise ValueError("one reference slot per pair of the batch")
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_set_ref_slots(self._h, arr.ctypes.data))

    def promote(self, slot: int):
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_promote(self._h, int(slot)))

    def retrack(self):
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_retrack(self._h))

    def host_bytes(self):
        """(H2D, D2H) bytes one submit_host / wait_host pair moves (only the LUT-reachable part of the images is uploaded)."""
        a, b = C.c_int64(), C.c_int64()
        check(self.ctx.lib.sos_frontend_host_bytes(self._h, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def step_host(self, *inputs):
        return self.wait_host(self.submit_host(*inputs))

    # -- images-in steps (sos_frontend_set_detector) -------------------------------------------------------------------
    def set_detector(self, masks_top, masks_bot, corners_per_bucket: int, quality_level: float = 0.01,
                     min_distance: float = 5.0, median: bool = True):
        """Detect the features inside the step, as features.FeatureFront does: masks uint8 [n_buckets, pano_rows,
        pano_cols] per view (numpy or torch), goodFeaturesToTrack(maxCorners = corners_per_bucket, quality_level,
        min_distance) per mask after an optional 11 x 11 median, then ORB description."""
        self._need(False, "set_detector")
        c = self.cfg
        ms = []
        for name, m in (("masks_top", masks_top), ("masks_bot", masks_bot)):
            t = (m if isinstance(m, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(m))).to(self.ctx.device)
            if tuple(t.shape) != (c.n_buckets, c.pano_rows, c.pano_cols):
                raise ValueError(f"{name} must be [n_buckets, pano_rows, pano_cols]")
            ms.append(t.contiguous())
        d = _DetectConfig(int(corners_per_bucket), int(bool(median)), float(quality_level), float(min_distance))
        self.ctx._sync_stream()
        # the masks are packed into bits by the call, which returns after that: they need not outlive it
        check(self.ctx.lib.sos_frontend_set_detector(self._h, C.byref(d), *(self.ctx._t(m, torch.uint8, "masks") for m in ms)))

    def _check_omni(self, omni, on_device: bool):
        self._need(False, "step_images / submit_host_images")
        c = self.cfg
        shape = (c.batch, c.src_h, c.src_w, c.channels)
        if tuple(omni.shape) != shape:
            raise ValueError(f"omni: expected shape {shape}, got {tuple(omni.shape)}")
        if on_device:
            return self.ctx._t(omni, torch.uint8, "omni")
        if isinstance(omni, torch.Tensor):
            if omni.is_cuda or omni.dtype != torch.uint8 or not omni.is_contiguous():
                raise TypeError("omni: expected a contiguous host tensor of torch.uint8")
            return omni.data_ptr()
        if omni.dtype != np.uint8 or not omni.flags.c_contiguous:
            raise TypeError("omni: expected a C-contiguous host array of uint8")
        return omni.ctypes.data

    def step_images(self, omni):
        """Asynchronous images-in step on device omni [batch, src_h, src_w, 3]; results in `buffers()` / `features()`."""
        p = self._check_omni(omni, True)
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_step_images(self._h, p))

    def submit_host_images(self, omni) -> int:
        """Images-in step on host omni (pinned): only the LUT-reachable image bands go over PCIe.  -> ticket for wait_host."""
        p = self._check_omni(omni, False)
        t = C.c_int()
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_submit_host_images(self._h, p, C.byref(t)))
        return t.value

    def step_host_images(self, omni):
        return self.wait_host(self.submit_host_images(omni))

    def host_images_bytes(self) -> int:
        """H2D bytes of one submit_host_images: host_bytes() without the feature arrays."""
        self._need(False, "host_images_bytes")
        c = self.cfg
        h2d, _ = self.host_bytes()
        return h2d - c.batch * (2 * c.max_feat_per_view * (2 * 4 + 32) + 2 * (c.n_buckets + 1) * 4)

    def features(self) -> dict:
        """Zero-copy torch views of the features the last images-in step detected (layout of `step`'s inputs, desc as
        uint8 [batch, max_feat_per_view, 32]) and detect_stats int32 [batch, 2, 4] (valid until close())."""
        self._need(False, "features")
        f = _Features()
        check(self.ctx.lib.sos_frontend_get_features(self._h, C.byref(f)))
        c = self.cfg
        B, F, nb = c.batch, c.max_feat_per_view, c.n_buckets
        shapes = {"px_top": ((B, F, 2), "f32"), "desc_top": ((B, F, 32), "u8"), "boff_top": ((B, nb + 1), "i32"),
                  "px_bot": ((B, F, 2), "f32"), "desc_bot": ((B, F, 32), "u8"), "boff_bot": ((B, nb + 1), "i32"),
                  "detect_stats": ((B, 2, 4), "i32")}
        out = {}
        for name in _FEATURE_FIELDS:
            shape, kind = shapes[name]
            out[name] = torch.as_tensor(_DeviceArray(getattr(f, name), shape, _TYPES[kind][0], self), device=self.ctx.device)
        return out

    # -- RGB-D steps ---------------------------------------------------------------------------------------------------
    def _check_rgbd(self, depth, px, desc, n_kp, on_device: bool):
        self._need(True, "step_rgbd / submit_host_rgbd")
        c = self.cfg
        shapes = {"depth": ((c.batch, c.height, c.width), (torch.float32, np.float32)),
                  "px": ((c.batch, c.max_kp, 2), (torch.float32, np.float32)),
                  "desc": ((c.batch, c.max_kp, 32), (torch.uint8, np.uint8)),
                  "n_kp": ((c.batch,), (torch.int32, np.int32))}
        ptrs = []
        for k, v in (("depth", depth), ("px", px), ("desc", desc), ("n_kp", n_kp)):
            shape, (tdt, ndt) = shapes[k]
            if tuple(v.shape) != shape:
                raise ValueError(f"{k}: expected shape {shape}, got {tuple(v.shape)}")
            if on_device:
                ptrs.append(self.ctx._t(v, tdt, k))
                continue
            if isinstance(v, torch.Tensor):
                if v.is_cuda or v.dtype != tdt or not v.is_contiguous():
                    raise TypeError(f"{k}: expected a contiguous host tensor of {tdt}")
                ptrs.append(v.data_ptr())
            else:
                if v.dtype != ndt or not v.flags.c_contiguous:
                    raise TypeError(f"{k}: expected a C-contiguous host array of {ndt}")
                ptrs.append(v.ctypes.data)
            if k == "n_kp":
                # host path: the counts are at hand, so refuse what the device path can only clamp to [0, max_kp]
                n = np.asarray(v)
                if n.min() < 0 or n.max() > c.max_kp:
                    raise ValueError(f"n_kp must lie in [0, max_kp = {c.max_kp}], got [{int(n.min())}, {int(n.max())}]")
        return ptrs

    def step_rgbd(self, depth, px, desc, n_kp):
        """Asynchronous RGB-D step on device tensors: depth [batch, height, width] float32, px [batch, max_kp, 2] float32,
        desc [batch, max_kp, 32] uint8, n_kp [batch] int32 (read on the device and clamped to [0, max_kp]); results are
        read through `buffers()`."""
        p = self._check_rgbd(depth, px, desc, n_kp, True)
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_step_rgbd(self._h, *p))

    def submit_host_rgbd(self, depth, px, desc, n_kp) -> int:
        """RGB-D step on host arrays (pinned for full copy bandwidth; whole depth maps are uploaded).  -> ticket for
        wait_host."""
        p = self._check_rgbd(depth, px, desc, n_kp, False)
        t = C.c_int()
        self.ctx._sync_stream()
        check(self.ctx.lib.sos_frontend_submit_host_rgbd(self._h, *p, C.byref(t)))
        return t.value

    def step_host_rgbd(self, depth, px, desc, n_kp):
        return self.wait_host(self.submit_host_rgbd(depth, px, desc, n_kp))

    def buffers(self) -> dict:
        """Zero-copy torch views of the device buffers (valid until close()).  An RGB-D front-end has one view and no
        panorama / stereo / second-view / camera-index / overflow buffers (they are absent from the dict)."""
        b = _Buffers()
        check(self.ctx.lib.sos_frontend_get_buffers(self._h, C.byref(b)))
        c = self.cfg
        V = int(b.views)
        B, cap, slots = c.batch, int(b.cap), c.batch + 1
        F, S = (0, 0) if self.rgbd else (c.max_feat_per_view, c.batch * c.n_buckets)
        shapes = {
            "pano": None if self.rgbd else (B, 2, c.pano_rows, c.pano_cols, c.channels),
            "st_q_start": (S,), "st_q_len": (S,), "st_t_start": (S,), "st_t_len": (S,),
            "st_idx0": (B * F,), "st_d0": (B * F,), "st_pair_q": (B * F,), "st_pair_t": (B * F,), "st_pair_d": (B * F,),
            "st_pair_count": (S,), "uv_c": (V, slots * cap, 2), "uv_top": (slots, cap, 2), "uv_bot": (slots, cap, 2),
            "b_top": (slots, cap, 3), "b_bot": (slots, cap, 3), "xyz": (slots, cap, 3), "src_top": (slots, cap),
            "src_bot": (slots, cap), "n": (slots,), "desc_c": (V, slots, cap, 8),
            "tm_q_start": (V * B,), "tm_q_len": (V * B,), "tm_t_start": (V * B,), "tm_t_len": (V * B,),
            "tm_idx0": (V * slots * cap,), "tm_d0": (V * slots * cap,), "tm_pair_q": (V * slots * cap,),
            "tm_pair_t": (V * slots * cap,), "tm_pair_d": (V * slots * cap,), "tm_pair_count": (V * B,),
            "p_ref": (B, V * cap, 3), "p_cur": (B, V * cap, 3), "f_cur": (B, V * cap, 3), "cam": (B, V * cap),
            "n_corr": (B,), "n_corr_top": (B,), "ransac_pose": (B, 3, 4), "pose": (B, 3, 4), "best_hyp": (B,),
            "best_count": (B,), "n_refit": (B,), "inlier_mask": (B, V * cap), "stats": (B, 4), "refine_stats": (B, 4), "ref_slot": (B,),
            "overflow": (B,),
        }
        out = {}
        for name, kind in _BUF_FIELDS:
            if not getattr(b, name):
                continue
            typestr, _ = _TYPES[kind]
            out[name] = torch.as_tensor(_DeviceArray(getattr(b, name), shapes[name], typestr, self), device=self.ctx.device)
        out["launches_per_step"] = int(b.launches_per_step)
        return out
