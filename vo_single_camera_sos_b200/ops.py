"""Device-tensor front door to libsosfront.so.

Each function takes CUDA `torch.Tensor`s (PyTorch is only the allocator / stream provider), checks dtype, layout and
device, and passes raw pointers to the C-ABI declared in include/sosfront.h.  Work is enqueued on the current torch
stream of the context's device.  There is no CPU path: a missing library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C
import threading
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import SosError, check  # noqa: F401  (re-exported)

MATCH_NN, MATCH_RATIO, MATCH_CROSS = 0, 1, 2
SCORE_EUCLID, SCORE_BEARING = 0, 1
SOLVER_ARUN, SOLVER_P3P = 0, 1
L2F_STATS, L2F_STAT_REDECIDED, L2F_STAT_BAND_PPM = 2, 0, 1   # sosfront.h SOS_L2F_*
REFINE_NONE, REFINE_ARUN, REFINE_LM = 0, 1, 2

GUM_FIELDS = ("xi1", "xi2", "xi3", "k1", "k2", "k3", "gamma1", "gamma2", "alpha_c", "u_center", "v_center",
              "l1", "l2", "l3", "p1", "p2", "plane_k", "use_distortion")
PANO_FIELDS = ("cols", "rows", "pixel_size", "cyl_height_max", "cyl_circumference", "cyl_radius")
RGBD_FIELDS = ("fx", "fy", "center_x", "center_y", "focal_length_m", "depth_is_Z")


def _darr(values: Sequence[float], n: int, what: str):
    a = np.ascontiguousarray(np.asarray(values, dtype=np.float64).reshape(-1))
    if a.size != n:
        raise ValueError(f"{what}: expected {n} doubles, got {a.size}")
    return a


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


class Context:
    """One libsosfront context = one device + the current torch stream. Not thread-safe; make one per thread."""

    def __init__(self, device: int | torch.device | None = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("vo_single_camera_sos_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
        h = C.c_void_p()
        check(self.lib.sos_ctx_create(self.device.index or 0, C.byref(h)))
        self._h = h
        self._stream_ptr = None
        self._sync_stream()

    def close(self):
        if getattr(self, "_h", None):
            self.lib.sos_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing -------------------------------------------------------------------------------------------
    def _sync_stream(self):
        s = torch.cuda.current_stream(self.device).cuda_stream
        if s != self._stream_ptr:
            check(self.lib.sos_ctx_set_stream(self._h, C.c_void_p(s)))  # 0 = legacy default stream
            self._stream_ptr = s

    def reserve(self, nbytes: int):
        check(self.lib.sos_ctx_reserve(self._h, int(nbytes)))

    @property
    def launch_count(self) -> int:
        return int(self.lib.sos_ctx_launch_count(self._h))

    def _t(self, t: Optional[torch.Tensor], dtype, what: str, optional: bool = False):
        if t is None:
            if optional:
                return None
            raise ValueError(f"{what} is required")
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise TypeError(f"{what} must be a CUDA tensor (no CPU fallback)")
        if t.device != self.device:
            raise ValueError(f"{what} lives on {t.device}, context is on {self.device}")
        if t.dtype != dtype:
            raise TypeError(f"{what} must be {dtype}, got {t.dtype}")
        if not t.is_contiguous():
            raise ValueError(f"{what} must be contiguous")
        return t.data_ptr()

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    # -- step 1: remap ----------------------------------------------------------------------------------------
    def lut_pack(self, map_x: torch.Tensor, map_y: torch.Tensor, src_hw, mask: Optional[torch.Tensor] = None):
        """map_x/map_y [rows, cols] float32 or float64 -> packed LUT [rows, cols] int64 (bit pattern of uint64)."""
        self._sync_stream()
        if map_x.shape != map_y.shape or map_x.dim() != 2:
            raise ValueError("map_x / map_y must be 2-D and of equal shape")
        rows, cols = map_x.shape
        h, w = int(src_hw[0]), int(src_hw[1])
        if mask is not None and tuple(mask.shape) != (h, w):
            raise ValueError("mask must have the source image shape")
        lut = self.empty((rows, cols), torch.int64)
        fn = self.lib.sos_lut_pack_f64 if map_x.dtype == torch.float64 else self.lib.sos_lut_pack_f32
        check(fn(self._h, self._t(map_x, map_x.dtype, "map_x"), self._t(map_y, map_x.dtype, "map_y"), rows, cols,
                 self._t(mask, torch.uint8, "mask", optional=True), h, w, lut.data_ptr()))
        return lut

    def remap(self, src: torch.Tensor, lut: torch.Tensor, border=(0, 0, 0, 0), background=(0, 0, 0, 0),
              out: Optional[torch.Tensor] = None):
        """src [B,H,W,C] (or [B,H,W]) uint8, lut [V,rows,cols] int64 -> dst [B,V,rows,cols,C] uint8."""
        self._sync_stream()
        squeeze = src.dim() == 3
        if squeeze:
            src = src.unsqueeze(-1)
        if lut.dim() == 2:
            lut = lut.unsqueeze(0)
        b, h, w, ch = src.shape
        v, rows, cols = lut.shape
        if out is None:
            out = self.empty((b, v, rows, cols, ch), torch.uint8)
        elif tuple(out.shape) != (b, v, rows, cols, ch):
            raise ValueError("out has the wrong shape")
        bd = np.zeros(4, np.uint8)
        bg = np.zeros(4, np.uint8)
        bd[:ch] = np.asarray(border, np.uint8).reshape(-1)[:ch]
        bg[:ch] = np.asarray(background, np.uint8).reshape(-1)[:ch]
        check(self.lib.sos_remap_u8(self._h, self._t(src, torch.uint8, "src"), b, h, w, ch,
                                    self._t(lut, torch.int64, "lut"), v, rows, cols, _ptr(bd), _ptr(bg),
                                    self._t(out, torch.uint8, "out")))
        return out[..., 0] if squeeze else out

    def gum_project(self, gum, pts: torch.Tensor):
        self._sync_stream()
        g = _darr(gum, len(GUM_FIELDS), "gum")
        n = pts.shape[0]
        uv = self.empty((n, 2), torch.float64)
        check(self.lib.sos_gum_project(self._h, _ptr(g), self._t(pts, torch.float64, "pts"), n, uv.data_ptr()))
        return uv

    def lut_build(self, gum, rows: int, cols: int, cyl_height_max: float, cyl_height_min: float, elev_lo: float,
                  elev_hi: float):
        self._sync_stream()
        g = _darr(gum, len(GUM_FIELDS), "gum")
        mx = self.empty((rows, cols), torch.float64)
        my = self.empty((rows, cols), torch.float64)
        check(self.lib.sos_lut_build(self._h, _ptr(g), rows, cols, float(cyl_height_max), float(cyl_height_min),
                                     float(elev_lo), float(elev_hi), mx.data_ptr(), my.data_ptr()))
        return mx, my

    # -- step 2: Hamming ----------------------------------------------------------------------------------------
    def hamming_top2(self, q: torch.Tensor, t: torch.Tensor, q_start, q_len, t_start, t_len, max_nq: int, max_nt: int,
                     want_second: bool = True, out=None):
        """q [Nq,32] uint8 (or [Nq,8] int32), t likewise; q_start/q_len/t_start/t_len [S] int32 DEVICE tensors."""
        self._sync_stream()
        nq = q.shape[0]
        n_seg = q_start.numel()
        qp = self._desc(q, "q")
        tp = self._desc(t, "t")
        if out is None:
            idx0 = torch.full((nq,), -1, dtype=torch.int32, device=self.device)
            d0 = torch.full((nq,), -1, dtype=torch.int32, device=self.device)
            idx1 = torch.full((nq,), -1, dtype=torch.int32, device=self.device) if want_second else None
            d1 = torch.full((nq,), -1, dtype=torch.int32, device=self.device) if want_second else None
        else:
            idx0, d0, idx1, d1 = out
        check(self.lib.sos_hamming_top2(self._h, qp, tp, self._t(q_start, torch.int32, "q_start"),
                                        self._t(q_len, torch.int32, "q_len"), self._t(t_start, torch.int32, "t_start"),
                                        self._t(t_len, torch.int32, "t_len"), n_seg, int(max_nq), int(max_nt),
                                        idx0.data_ptr(), d0.data_ptr(),
                                        idx1.data_ptr() if idx1 is not None else None,
                                        d1.data_ptr() if d1 is not None else None))
        return idx0, d0, idx1, d1

    def l2_top2(self, q: torch.Tensor, t: torch.Tensor, q_start, q_len, t_start, t_len, max_nq: int, max_nt: int,
                want_second: bool = True):
        """Float descriptors (integer-valued in [0, 255], e.g. cv2 SIFT): q [Nq, dim], t [Nt, dim] float32, dim <= 128.
        -> (idx0 int32, d0 float32, idx1, d1) like hamming_top2, distances = cv2's NORM_L2.  Raises ValueError when a
        descriptor value is not an integer in [0, 255] (the tensor-core path is exact only for those)."""
        self._sync_stream()
        nq, dim = q.shape
        if t.dim() != 2 or t.shape[1] != dim or dim > 128:
            raise ValueError("q / t must be [N, dim] with the same dim <= 128")
        n_seg = q_start.numel()
        idx0 = torch.full((nq,), -1, dtype=torch.int32, device=self.device)
        d0 = torch.full((nq,), -1.0, dtype=torch.float32, device=self.device)
        idx1 = torch.full((nq,), -1, dtype=torch.int32, device=self.device) if want_second else None
        d1 = torch.full((nq,), -1.0, dtype=torch.float32, device=self.device) if want_second else None
        flag = torch.zeros((1,), dtype=torch.int32, device=self.device)
        check(self.lib.sos_l2_top2(self._h, self._t(q, torch.float32, "q"), self._t(t, torch.float32, "t"), int(dim),
                                   self._t(q_start, torch.int32, "q_start"), self._t(q_len, torch.int32, "q_len"),
                                   self._t(t_start, torch.int32, "t_start"), self._t(t_len, torch.int32, "t_len"), n_seg,
                                   int(max_nq), int(max_nt), idx0.data_ptr(), d0.data_ptr(),
                                   idx1.data_ptr() if idx1 is not None else None, d1.data_ptr() if d1 is not None else None,
                                   flag.data_ptr()))
        if int(flag.item()):
            raise ValueError("float descriptors must hold integers in [0, 255] (cv2 SIFT); other values are not supported "
                             "by the exact tensor-core L2 matcher")
        return idx0, d0, idx1, d1

    def l2f_top2(self, q: torch.Tensor, t: torch.Tensor, q_start, q_len, t_start, t_len, max_nq: int, max_nt: int,
                 want_second: bool = True, stats: Optional[torch.Tensor] = None):
        """Any finite float descriptors (SURF, KAZE, RootSIFT, ...): q [Nq, dim], t [Nt, dim] float32, 1 <= dim <= 128.
        -> (idx0 int32, d0 float32, idx1, d1) like l2_top2, equal bit for bit to a float64 reference: d^2 summed over k in
        order without FMA, ties to the lowest train row, distance = float32(sqrt(d^2)).  Raises ValueError on NaN / Inf.
        stats: optional DEVICE int32 [L2F_STATS] -> queries re-decided in float64, largest error / band in ppm."""
        self._sync_stream()
        nq, dim = q.shape
        if t.dim() != 2 or t.shape[1] != dim or not 1 <= dim <= 128:
            raise ValueError("q / t must be [N, dim] with the same 1 <= dim <= 128")
        if stats is not None and stats.numel() < L2F_STATS:
            raise ValueError(f"stats needs {L2F_STATS} int32 entries")
        n_seg = q_start.numel()
        idx0 = torch.full((nq,), -1, dtype=torch.int32, device=self.device)
        d0 = torch.full((nq,), -1.0, dtype=torch.float32, device=self.device)
        idx1 = torch.full((nq,), -1, dtype=torch.int32, device=self.device) if want_second else None
        d1 = torch.full((nq,), -1.0, dtype=torch.float32, device=self.device) if want_second else None
        flag = torch.zeros((1,), dtype=torch.int32, device=self.device)
        check(self.lib.sos_l2f_top2(self._h, self._t(q, torch.float32, "q"), self._t(t, torch.float32, "t"), int(dim),
                                    self._t(q_start, torch.int32, "q_start"), self._t(q_len, torch.int32, "q_len"),
                                    self._t(t_start, torch.int32, "t_start"), self._t(t_len, torch.int32, "t_len"), n_seg,
                                    int(max_nq), int(max_nt), idx0.data_ptr(), d0.data_ptr(),
                                    idx1.data_ptr() if idx1 is not None else None, d1.data_ptr() if d1 is not None else None,
                                    flag.data_ptr(), self._t(stats, torch.int32, "stats", optional=True)))
        if int(flag.item()):
            raise ValueError("float descriptors must be finite (a value is NaN or Inf)")
        return idx0, d0, idx1, d1

    def hamming_radius(self, q: torch.Tensor, t: torch.Tensor, max_distance: int):
        """Every (query, train, distance) with distance <= max_distance, query-major, train index ascending within a query
        (cv2.BFMatcher.radiusMatch).  -> (query int64 [M], train int32 [M], distance int32 [M]) device tensors."""
        self._sync_stream()
        nq, nt = q.shape[0], t.shape[0]
        qp, tp = self._desc(q, "q"), self._desc(t, "t")
        count = torch.zeros((nq,), dtype=torch.int32, device=self.device)
        check(self.lib.sos_hamming_radius(self._h, qp, nq, tp, nt, int(max_distance), count.data_ptr(), None, None, None))
        incl = torch.cumsum(count.to(torch.int64), 0)
        offset = (incl - count).contiguous()
        m = int(incl[-1]) if nq else 0
        out_t = torch.empty((max(m, 1),), dtype=torch.int32, device=self.device)
        out_d = torch.empty((max(m, 1),), dtype=torch.int32, device=self.device)
        if m:
            check(self.lib.sos_hamming_radius(self._h, qp, nq, tp, nt, int(max_distance), None, offset.data_ptr(),
                                              out_t.data_ptr(), out_d.data_ptr()))
        qi = torch.repeat_interleave(torch.arange(nq, device=self.device), count.to(torch.int64))
        return qi, out_t[:m], out_d[:m]

    def _desc(self, d: torch.Tensor, what: str):
        if d.dtype == torch.uint8:
            if d.dim() != 2 or d.shape[1] != 32:
                raise ValueError(f"{what}: uint8 descriptors must be [N,32]")
            return self._t(d, torch.uint8, what)
        if d.dim() != 2 or d.shape[1] != 8:
            raise ValueError(f"{what}: int32 descriptors must be [N,8]")
        return self._t(d, torch.int32, what)

    def match_select(self, mode: int, idx0, d0, d1, q_start, q_len, t_start, rev_idx0=None, px_q=None, px_t=None,
                     max_du: float = -1.0, min_dv: float = -1.0, ratio: float = 0.75, out=None):
        self._sync_stream()
        nq = idx0.shape[0]
        n_seg = q_start.numel()
        if out is None:
            out_q = self.empty((nq,), torch.int32)
            out_t = self.empty((nq,), torch.int32)
            out_d = self.empty((nq,), torch.int32)
            out_count = self.empty((n_seg,), torch.int32)
        else:
            out_q, out_t, out_d, out_count = out
        check(self.lib.sos_match_select(
            self._h, int(mode), float(ratio), self._t(idx0, torch.int32, "idx0"), self._t(d0, torch.int32, "d0"),
            self._t(d1, torch.int32, "d1", optional=True), self._t(rev_idx0, torch.int32, "rev_idx0", optional=True),
            self._t(q_start, torch.int32, "q_start"), self._t(q_len, torch.int32, "q_len"),
            self._t(t_start, torch.int32, "t_start"), n_seg,
            self._t(px_q, torch.float32, "px_q", optional=True), self._t(px_t, torch.float32, "px_t", optional=True),
            float(max_du), float(min_dv), out_q.data_ptr(), out_t.data_ptr(), out_d.data_ptr(), out_count.data_ptr()))
        return out_q, out_t, out_d, out_count

    # -- steps 3+4 ----------------------------------------------------------------------------------------------
    def lift_pano(self, pano, uv: torch.Tensor, want_bearing: bool = True):
        self._sync_stream()
        p = _darr(pano, len(PANO_FIELDS), "pano")
        n = uv.shape[0]
        az = self.empty((n,), torch.float32)
        el = self.empty((n,), torch.float32)
        bearing = self.empty((n, 3), torch.float32) if want_bearing else None
        check(self.lib.sos_lift_pano(self._h, _ptr(p), self._t(uv, torch.float32, "uv"), n, az.data_ptr(), el.data_ptr(),
                                     bearing.data_ptr() if want_bearing else None))
        return az, el, bearing

    def lift_pano_f64(self, pano, uv: torch.Tensor):
        """float64 in / out variant of lift_pano (the reference's dtype)."""
        self._sync_stream()
        p = _darr(pano, len(PANO_FIELDS), "pano")
        n = uv.shape[0]
        az = self.empty((n,), torch.float64)
        el = self.empty((n,), torch.float64)
        bearing = self.empty((n, 3), torch.float64)
        check(self.lib.sos_lift_pano_f64(self._h, _ptr(p), self._t(uv, torch.float64, "uv"), n, az.data_ptr(),
                                         el.data_ptr(), bearing.data_ptr()))
        return az, el, bearing

    def angles_to_sphere_f64(self, az: torch.Tensor, el: torch.Tensor):
        self._sync_stream()
        n = az.shape[0]
        out = self.empty((n, 3), torch.float64)
        check(self.lib.sos_angles_to_sphere_f64(self._h, self._t(az, torch.float64, "az"), self._t(el, torch.float64, "el"),
                                                n, out.data_ptr()))
        return out

    def range_gate(self, xyz: torch.Tensor, rmin: float, rmax: float, homogeneous_norm: bool):
        self._sync_stream()
        n = xyz.shape[0]
        valid = self.empty((n,), torch.uint8)
        check(self.lib.sos_range_gate_f64(self._h, self._t(xyz, torch.float64, "xyz"), n, float(rmin), float(rmax),
                                          int(bool(homogeneous_norm)), valid.data_ptr()))
        return valid

    def triangulate_midpoint_f64(self, az1, el1, az2, el2, f1, f2, rmin: float = 0.0, rmax: float = 0.0,
                                 homogeneous_norm: bool = False):
        self._sync_stream()
        n = az1.shape[0]
        a = _darr(f1, 3, "f1")
        b = _darr(f2, 3, "f2")
        xyz = self.empty((n, 3), torch.float64)
        valid = self.empty((n,), torch.uint8)
        check(self.lib.sos_triangulate_midpoint_f64(
            self._h, self._t(az1, torch.float64, "az1"), self._t(el1, torch.float64, "el1"),
            self._t(az2, torch.float64, "az2"), self._t(el2, torch.float64, "el2"), n, _ptr(a), _ptr(b), float(rmin),
            float(rmax), int(bool(homogeneous_norm)), xyz.data_ptr(), valid.data_ptr()))
        return xyz, valid

    # -- N3: feature description ---------------------------------------------------------------------------------
    def median_blur_11(self, img: torch.Tensor) -> torch.Tensor:
        """cv2.medianBlur(img, 11): uint8 [H, W], [H, W, 3], [n, H, W] (gray batch is [n, H, W, 1]) or [n, H, W, 3]."""
        self._sync_stream()
        if img.dim() == 2:
            x = img[None, :, :, None]
        elif img.dim() == 3:
            x = img[None] if img.shape[-1] == 3 else img[..., None]
        else:
            x = img
        n, H, W, ch = x.shape
        out = self.empty((n, H, W, ch), torch.uint8)
        check(self.lib.sos_median_blur_11(self._h, self._t(x, torch.uint8, "img"), n, H, W, ch, out.data_ptr()))
        return out.reshape(img.shape)

    def median_blur_11_gray(self, bgr: torch.Tensor, want_bgr: bool = False):
        """cv2.cvtColor(cv2.medianBlur(bgr, 11), COLOR_BGR2GRAY) in one kernel: uint8 [n, H, W, 3] -> gray [n, H, W]
        (and the blurred BGR image when want_bgr)."""
        self._sync_stream()
        n, H, W, ch = bgr.shape
        assert ch == 3
        gray = self.empty((n, H, W), torch.uint8)
        out = self.empty((n, H, W, 3), torch.uint8) if want_bgr else None
        check(self.lib.sos_median_blur_11_gray(self._h, self._t(bgr, torch.uint8, "bgr"), n, H, W,
                                               out.data_ptr() if want_bgr else None, gray.data_ptr()))
        return (gray, out) if want_bgr else gray

    def bgr_to_gray(self, bgr: torch.Tensor) -> torch.Tensor:
        """uint8 [..., 3] -> uint8 [...]  (cv2.COLOR_BGR2GRAY, bit-exact)."""
        self._sync_stream()
        if bgr.shape[-1] != 3:
            raise ValueError("expected a [..., 3] BGR image")
        gray = self.empty(tuple(bgr.shape[:-1]), torch.uint8)
        check(self.lib.sos_bgr_to_gray(self._h, self._t(bgr, torch.uint8, "bgr"), gray.numel(), gray.data_ptr()))
        return gray

    def orb_blur(self, gray: torch.Tensor) -> torch.Tensor:
        self._sync_stream()
        g = gray[None] if gray.dim() == 2 else gray
        out = self.empty(tuple(g.shape), torch.uint8)
        check(self.lib.sos_orb_blur(self._h, self._t(g, torch.uint8, "gray"), g.shape[0], g.shape[1], g.shape[2], out.data_ptr()))
        return out[0] if gray.dim() == 2 else out

    def orb_describe(self, gray: torch.Tensor, kp_xy: torch.Tensor, kp_angle_deg=None, kp_image=None):
        """gray uint8 [H, W] or [n_images, H, W]; kp_xy float32 [n, 2] -> (desc uint8 [n, 32], keep uint8 [n])."""
        self._sync_stream()
        g = gray[None] if gray.dim() == 2 else gray
        n = kp_xy.shape[0]
        desc = self.empty((n, 32), torch.uint8)
        keep = self.empty((n,), torch.uint8)
        check(self.lib.sos_orb_describe(
            self._h, self._t(g, torch.uint8, "gray"), g.shape[0], g.shape[1], g.shape[2], self._t(kp_xy, torch.float32, "kp_xy"),
            None if kp_angle_deg is None else self._t(kp_angle_deg, torch.float32, "kp_angle_deg"),
            None if kp_image is None else self._t(kp_image, torch.int32, "kp_image"), n, desc.data_ptr(), keep.data_ptr()))
        return desc, keep

    def corner_min_eigenval(self, gray: torch.Tensor) -> torch.Tensor:
        self._sync_stream()
        g = gray[None] if gray.dim() == 2 else gray
        eig = self.empty(tuple(g.shape), torch.float32)
        check(self.lib.sos_corner_min_eigenval(self._h, self._t(g, torch.uint8, "gray"), g.shape[0], g.shape[1], g.shape[2],
                                               eig.data_ptr()))
        return eig[0] if gray.dim() == 2 else eig

    def gft_detect(self, gray: torch.Tensor, masks, max_corners: int, quality_level: float = 0.01, min_distance: float = 5.0,
                   want_eig: bool = False):
        """cv2.goodFeaturesToTrack for every (image, mask): gray uint8 [n, H, W] (or [H, W]), masks uint8 [m, H, W] or None
        -> xy float32 [n, m, max_corners, 2] (strongest first), count int32 [n, m] (and eig float32 [n, H, W])."""
        self._sync_stream()
        g = gray[None] if gray.dim() == 2 else gray
        n, H, W = g.shape
        m = 1 if masks is None else masks.shape[0]
        xy = self.empty((n, m, max_corners, 2), torch.float32)
        count = self.empty((n, m), torch.int32)
        eig = self.empty((n, H, W), torch.float32) if want_eig else None
        check(self.lib.sos_gft_detect(
            self._h, self._t(g, torch.uint8, "gray"), None if masks is None else self._t(masks, torch.uint8, "masks"), n, H, W,
            m, int(max_corners), float(quality_level), float(min_distance), xy.data_ptr(), count.data_ptr(),
            None if eig is None else eig.data_ptr()))
        return (xy, count, eig) if want_eig else (xy, count)

    def dense_triangulate(self, pano_top, pano_bot, disparity: torch.Tensor, f1, f2, min_disparity: float = 1.0,
                          max_disparity: float = 0.0, lowest_reference_row: float = float("inf"), roi_cols=None, out=None):
        """Disparity maps float32 [n, rows, cols] (or [rows, cols]) -> xyz float32 [..., rows, cols, 3] (NaN = invalid),
        valid uint8 [..., rows, cols]  (sos_dense_triangulate)."""
        self._sync_stream()
        squeeze = disparity.dim() == 2
        d = disparity[None] if squeeze else disparity
        n, rows, cols = d.shape
        pt, pb = _darr(pano_top, 6, "pano_top"), _darr(pano_bot, 6, "pano_bot")
        a, b = _darr(f1, 3, "f1"), _darr(f2, 3, "f2")
        xyz, valid = out if out is not None else (self.empty((n, rows, cols, 3), torch.float32),
                                                  self.empty((n, rows, cols), torch.uint8))
        r0, r1 = (-1, -1) if roi_cols is None else (int(roi_cols[0]), int(roi_cols[1]))
        check(self.lib.sos_dense_triangulate(
            self._h, _ptr(pt), _ptr(pb), self._t(d, torch.float32, "disparity"), n, rows, cols, float(min_disparity),
            float(max_disparity), float(lowest_reference_row), r0, r1, _ptr(a), _ptr(b), xyz.data_ptr(), valid.data_ptr()))
        return (xyz[0], valid[0]) if squeeze and out is None else (xyz, valid)

    def lift_gum(self, gum, uv: torch.Tensor):
        self._sync_stream()
        g = _darr(gum, len(GUM_FIELDS), "gum")
        n = uv.shape[0]
        sphere = self.empty((n, 3), torch.float64)
        az = self.empty((n,), torch.float64)
        el = self.empty((n,), torch.float64)
        check(self.lib.sos_lift_gum(self._h, _ptr(g), self._t(uv, torch.float64, "uv"), n, sphere.data_ptr(),
                                    az.data_ptr(), el.data_ptr()))
        return sphere, az, el

    def triangulate_midpoint(self, az1, el1, az2, el2, f1, f2, rmin: float = 0.0, rmax: float = 0.0,
                             homogeneous_norm: bool = False):
        self._sync_stream()
        n = az1.shape[0]
        a = _darr(f1, 3, "f1")
        b = _darr(f2, 3, "f2")
        xyz = self.empty((n, 3), torch.float32)
        valid = self.empty((n,), torch.uint8)
        check(self.lib.sos_triangulate_midpoint(
            self._h, self._t(az1, torch.float32, "az1"), self._t(el1, torch.float32, "el1"),
            self._t(az2, torch.float32, "az2"), self._t(el2, torch.float32, "el2"), n, _ptr(a), _ptr(b), float(rmin),
            float(rmax), int(bool(homogeneous_norm)), xyz.data_ptr(), valid.data_ptr()))
        return xyz, valid

    def stereo_lift_triangulate(self, pano_top, pano_bot, px_top, px_bot, pair_q, pair_t, pair_count, seg_off,
                                n_frames: int, segs_per_frame: int, f1, f2, rmin: float, rmax: float, cap_per_frame: int,
                                homogeneous_norm: bool = True, out: Optional[dict] = None,
                                max_pairs_per_seg: Optional[int] = None):
        self._sync_stream()
        pt = _darr(pano_top, len(PANO_FIELDS), "pano_top")
        pb = _darr(pano_bot, len(PANO_FIELDS), "pano_bot")
        a = _darr(f1, 3, "f1")
        b = _darr(f2, 3, "f2")
        rows = n_frames * cap_per_frame
        if out is None:
            out = {
                "uv_top": self.empty((rows, 2), torch.float32), "uv_bot": self.empty((rows, 2), torch.float32),
                "b_top": self.empty((rows, 3), torch.float32), "b_bot": self.empty((rows, 3), torch.float32),
                "xyz": self.empty((rows, 3), torch.float32), "src_top": self.empty((rows,), torch.int32),
                "src_bot": self.empty((rows,), torch.int32), "n": self.empty((n_frames,), torch.int32),
            }
        check(self.lib.sos_stereo_lift_triangulate(
            self._h, _ptr(pt), _ptr(pb), self._t(px_top, torch.float32, "px_top"),
            self._t(px_bot, torch.float32, "px_bot"), self._t(pair_q, torch.int32, "pair_q"),
            self._t(pair_t, torch.int32, "pair_t"), self._t(pair_count, torch.int32, "pair_count"),
            self._t(seg_off, torch.int32, "seg_off"), int(n_frames), int(segs_per_frame),
            int(max_pairs_per_seg if max_pairs_per_seg is not None else pair_q.shape[0]), int(pair_q.shape[0]), _ptr(a), _ptr(b),
            float(rmin), float(rmax), int(bool(homogeneous_norm)), int(cap_per_frame),
            out["uv_top"].data_ptr(), out["uv_bot"].data_ptr(), out["b_top"].data_ptr(), out["b_bot"].data_ptr(),
            out["xyz"].data_ptr(), out["src_top"].data_ptr(), out["src_bot"].data_ptr(), out["n"].data_ptr()))
        return out

    def rgbd_depth_to_z(self, cam, depth: torch.Tensor):
        self._sync_stream()
        c = _darr(cam, len(RGBD_FIELDS), "cam")
        d3 = depth if depth.dim() == 3 else depth.unsqueeze(0)
        b, h, w = d3.shape
        z = torch.empty_like(d3)
        check(self.lib.sos_rgbd_depth_to_z(self._h, _ptr(c), self._t(d3, torch.float32, "depth"), b, h, w, z.data_ptr()))
        return z if depth.dim() == 3 else z[0]

    def rgbd_backproject(self, cam, depth: torch.Tensor, u: torch.Tensor, v: torch.Tensor, zmin: float = 0.0,
                         zmax: float = 0.0):
        self._sync_stream()
        c = _darr(cam, len(RGBD_FIELDS), "cam")
        d3 = depth if depth.dim() == 3 else depth.unsqueeze(0)
        u2 = u if u.dim() == 2 else u.unsqueeze(0)
        v2 = v if v.dim() == 2 else v.unsqueeze(0)
        b, h, w = d3.shape
        n = u2.shape[1]
        xyz = self.empty((b, n, 3), torch.float32)
        bearing = self.empty((b, n, 3), torch.float32)
        valid = self.empty((b, n), torch.uint8)
        check(self.lib.sos_rgbd_backproject(self._h, _ptr(c), self._t(d3, torch.float32, "depth"), b, h, w,
                                            self._t(u2, torch.int32, "u"), self._t(v2, torch.int32, "v"), n,
                                            float(zmin), float(zmax), xyz.data_ptr(), bearing.data_ptr(),
                                            valid.data_ptr()))
        if depth.dim() == 2:
            return xyz[0], bearing[0], valid[0]
        return xyz, bearing, valid

    # -- step 5 -------------------------------------------------------------------------------------------------
    def arun_batch(self, v0: torch.Tensor, v1: torch.Tensor, with_scale: bool = False):
        """v0, v1 [n_sets, k, 3] float64 -> M [n_sets, 3, 4] float64, ok [n_sets] uint8."""
        self._sync_stream()
        n_sets, k, _ = v0.shape
        M = self.empty((n_sets, 3, 4), torch.float64)
        ok = self.empty((n_sets,), torch.uint8)
        check(self.lib.sos_arun_batch(self._h, self._t(v0, torch.float64, "v0"), self._t(v1, torch.float64, "v1"),
                                      n_sets, k, int(bool(with_scale)), M.data_ptr(), ok.data_ptr()))
        return M, ok

    def pixel_gate(self, pts_top: torch.Tensor, pts_bot: torch.Tensor, max_du: float, min_dv: float):
        """pts_* [n,2] float64 -> valid [n] uint8 (common_cv.filter_pixel_correspondences)."""
        self._sync_stream()
        n = pts_top.shape[0]
        valid = self.empty((n,), torch.uint8)
        check(self.lib.sos_pixel_gate(self._h, self._t(pts_top, torch.float64, "pts_top"),
                                      self._t(pts_bot, torch.float64, "pts_bot"), n, float(max_du), float(min_dv),
                                      valid.data_ptr()))
        return valid

    @staticmethod
    def _rig(rig, n_cams):
        if rig is None:
            return None, 0
        r = np.ascontiguousarray(np.asarray(rig, dtype=np.float64).reshape(-1))
        if r.size != 12 * n_cams:
            raise ValueError("rig must hold n_cams row-major 3x4 [Rc|tc] blocks")
        return r, n_cams

    def ransac_p3d(self, p_ref, p_cur, n, hyp, score_mode: int, threshold: float, f_cur=None, cam=None, rig=None,
                   n_cams: int = 0, hyp_offset: int = 0, want_mask: bool = True, all_counts=None):
        """p_ref, p_cur, f_cur [B, cap, 3] float32; cam [B, cap] uint8; n [B] int32; hyp [H,3] int64/uint32 bits."""
        self._sync_stream()
        B, cap, _ = p_ref.shape
        H = hyp.shape[0]
        r, n_cams = self._rig(rig, n_cams)
        pose = self.empty((B, 3, 4), torch.float32)
        best_hyp = self.empty((B,), torch.int32)
        best_count = self.empty((B,), torch.int32)
        mask = self.empty((B, cap), torch.uint8) if want_mask else None
        key = self.empty((B,), torch.int64)
        check(self.lib.sos_ransac_p3d(
            self._h, self._t(p_ref, torch.float32, "p_ref"), self._t(p_cur, torch.float32, "p_cur"),
            self._t(f_cur, torch.float32, "f_cur", optional=True), self._t(cam, torch.uint8, "cam", optional=True),
            self._t(n, torch.int32, "n"), B, cap, _ptr(r), n_cams, self._t(hyp, torch.int32, "hyp"), H, int(hyp_offset),
            int(score_mode), float(threshold), pose.data_ptr(), best_hyp.data_ptr(), best_count.data_ptr(),
            mask.data_ptr() if want_mask else None, key.data_ptr(),
            self._t(all_counts, torch.int32, "all_counts", optional=True)))
        return pose, best_hyp, best_count, mask, key

    def ransac_score_probe(self, p_ref, p_cur, f_cur, n, hyp, threshold: float, cam=None, rig=None, n_cams: int = 0,
                           score_mode: int = 1, want_sn: bool = True, stats=None):
        """Diagnostics of the score engines (sos_ransac_score_probe).  want_sn: run on the tensor-core engine and dump its two
        accumulators per pair; otherwise the engine is the one ransac_p3d picks.  stats: an optional DEVICE int32 tensor of
        SOS_SCORE_STATS (8) entries that receives the deferred-path counters (include/sosfront.h, SOS_STAT_*).
        Returns (all_counts [B, H] int32, sn [B, H, ceil(cap / 128) * 128, 2] float32 or None)."""
        self._sync_stream()
        if not want_sn and stats is None:
            raise ValueError("ransac_score_probe needs want_sn or stats")
        B, cap, _ = p_ref.shape
        H = hyp.shape[0]
        r, n_cams = self._rig(rig, n_cams)
        pose = self.empty((B, 3, 4), torch.float32)
        best_hyp = self.empty((B,), torch.int32)
        best_count = self.empty((B,), torch.int32)
        counts = self.empty((B, H), torch.int32)
        sn = torch.zeros((B, H, (cap + 127) // 128 * 128, 2), dtype=torch.float32, device=self.device) if want_sn else None
        if stats is not None and stats.numel() != 8:
            raise ValueError("stats must hold SOS_SCORE_STATS = 8 int32 entries")
        check(self.lib.sos_ransac_score_probe(
            self._h, self._t(p_ref, torch.float32, "p_ref"), self._t(p_cur, torch.float32, "p_cur"),
            self._t(f_cur, torch.float32, "f_cur", optional=True), self._t(cam, torch.uint8, "cam", optional=True),
            self._t(n, torch.int32, "n"), B, cap, _ptr(r), n_cams, self._t(hyp, torch.int32, "hyp"), H, int(score_mode),
            float(threshold), pose.data_ptr(), best_hyp.data_ptr(), best_count.data_ptr(), counts.data_ptr(),
            sn.data_ptr() if want_sn else None, self._t(stats, torch.int32, "stats", optional=True)))
        return counts, sn

    def ransac_p3p(self, p_ref, f_cur, n, hyp, threshold: float, cam=None, rig=None, n_cams: int = 0, hyp_offset: int = 0,
                   want_mask: bool = True, all_counts=None):
        """Bearing-only RANSAC (sos_ransac_p3p): p_ref, f_cur [B, cap, 3] float32; hyp [H,4] uint32 bits."""
        self._sync_stream()
        B, cap, _ = p_ref.shape
        H = hyp.shape[0]
        assert hyp.shape[1] == 4, "four sample numbers per hypothesis"
        r, n_cams = self._rig(rig, n_cams)
        pose = self.empty((B, 3, 4), torch.float32)
        best_hyp = self.empty((B,), torch.int32)
        best_count = self.empty((B,), torch.int32)
        mask = self.empty((B, cap), torch.uint8) if want_mask else None
        key = self.empty((B,), torch.int64)
        check(self.lib.sos_ransac_p3p(
            self._h, self._t(p_ref, torch.float32, "p_ref"), self._t(f_cur, torch.float32, "f_cur"),
            self._t(cam, torch.uint8, "cam", optional=True), self._t(n, torch.int32, "n"), B, cap, _ptr(r), n_cams,
            self._t(hyp, torch.int32, "hyp"), H, int(hyp_offset), float(threshold), pose.data_ptr(), best_hyp.data_ptr(),
            best_count.data_ptr(), mask.data_ptr() if want_mask else None, key.data_ptr(),
            self._t(all_counts, torch.int32, "all_counts", optional=True)))
        return pose, best_hyp, best_count, mask, key

    def ransac_p3d_eval(self, p_ref, p_cur, n, hyp_row, score_mode: int, threshold: float, f_cur=None, cam=None,
                        rig=None, n_cams: int = 0):
        self._sync_stream()
        B, cap, _ = p_ref.shape
        r, n_cams = self._rig(rig, n_cams)
        pose = self.empty((B, 3, 4), torch.float32)
        count = self.empty((B,), torch.int32)
        mask = self.empty((B, cap), torch.uint8)
        check(self.lib.sos_ransac_p3d_eval(
            self._h, self._t(p_ref, torch.float32, "p_ref"), self._t(p_cur, torch.float32, "p_cur"),
            self._t(f_cur, torch.float32, "f_cur", optional=True), self._t(cam, torch.uint8, "cam", optional=True),
            self._t(n, torch.int32, "n"), B, cap, _ptr(r), n_cams, self._t(hyp_row, torch.int32, "hyp_row"),
            int(score_mode), float(threshold), pose.data_ptr(), count.data_ptr(), mask.data_ptr()))
        return pose, count, mask

    def refit_inliers(self, p_ref, p_cur, mask, n):
        self._sync_stream()
        B, cap, _ = p_ref.shape
        pose = self.empty((B, 3, 4), torch.float32)
        used = self.empty((B,), torch.int32)
        check(self.lib.sos_refit_inliers(self._h, self._t(p_ref, torch.float32, "p_ref"),
                                         self._t(p_cur, torch.float32, "p_cur"), self._t(mask, torch.uint8, "mask"),
                                         self._t(n, torch.int32, "n"), B, cap, pose.data_ptr(), used.data_ptr()))
        return pose, used

    def refine_pose(self, p_ref, f_cur, cam, mask, n, rig, pose_in, max_iters: int = 30, cluster_size: int = 0):
        """Levenberg-Marquardt refinement of the bearing residual on the masked rows (sos_refine_pose).
        Returns (pose float32 [B,3,4], pose64 float64 [B,3,4], stats float64 [B,4])."""
        self._sync_stream()
        B, cap, _ = p_ref.shape
        pose = self.empty((B, 3, 4), torch.float32)
        pose64 = self.empty((B, 3, 4), torch.float64)
        stats = self.empty((B, 4), torch.float64)
        rig_arr = None if rig is None else np.ascontiguousarray(np.asarray(rig, np.float64).reshape(-1, 12))
        check(self.lib.sos_refine_pose(
            self._h, self._t(p_ref, torch.float32, "p_ref"), self._t(f_cur, torch.float32, "f_cur"),
            None if cam is None else self._t(cam, torch.uint8, "cam"),
            None if mask is None else self._t(mask, torch.uint8, "mask"), self._t(n, torch.int32, "n"), B, cap,
            None if rig_arr is None else rig_arr.ctypes.data, 0 if rig_arr is None else len(rig_arr),
            self._t(pose_in, torch.float32, "pose_in"), int(max_iters), int(cluster_size), pose.data_ptr(),
            pose64.data_ptr(), stats.data_ptr()))
        return pose, pose64, stats

    # -- per-launch device timing (sos_ctx_profile_*) ------------------------------------------------------------
    def profile_begin(self):
        self._sync_stream()
        check(self.lib.sos_ctx_profile_begin(self._h))

    def profile_end(self, max_n: int = 4096):
        """-> list of (entry point name#launch index, milliseconds) in launch order."""
        names = C.create_string_buffer(64 * max_n)
        ms = (C.c_float * max_n)()
        n = C.c_int()
        check(self.lib.sos_ctx_profile_end(self._h, names, len(names), ms, max_n, C.byref(n)))
        nm = names.value.decode().split("\n")[: n.value]
        return [(nm[i], float(ms[i])) for i in range(n.value)]

    # -- roofline denominators -----------------------------------------------------------------------------------
    def peak_popc(self) -> float:
        self._sync_stream()
        v = C.c_double()
        check(self.lib.sos_peak_popc(self._h, C.byref(v)))
        return v.value

    def peak_dfma(self) -> float:
        self._sync_stream()
        v = C.c_double()
        check(self.lib.sos_peak_dfma(self._h, C.byref(v)))
        return v.value

    def peak_ffma(self) -> float:
        self._sync_stream()
        v = C.c_double()
        check(self.lib.sos_peak_ffma(self._h, C.byref(v)))
        return v.value

    def peak_ffma2(self) -> float:
        """TFLOP/s of packed fma.rn.f32x2 (FFMA2)."""
        self._sync_stream()
        v = C.c_double()
        check(self.lib.sos_peak_ffma2(self._h, C.byref(v)))
        return v.value

    def peak_tmem_read(self) -> float:
        """TB/s of tcgen05.ld over all SMs (tensor memory -> registers)."""
        self._sync_stream()
        v = C.c_double()
        check(self.lib.sos_peak_tmem_read(self._h, C.byref(v)))
        return v.value


_tls = threading.local()


def default_context(device: Optional[int] = None) -> Context:
    """Per-thread, per-device context (the reference's VO loop runs on its own thread, pose_est_tools.py:1725)."""
    if device is None:
        device = torch.cuda.current_device()
    cache = getattr(_tls, "ctx", None)
    if cache is None:
        cache = _tls.ctx = {}
    if device not in cache:
        cache[device] = Context(device)
    return cache[device]
