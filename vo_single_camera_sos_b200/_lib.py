"""ctypes binding of libsosfront.so (the C-ABI declared in include/sosfront.h).

There is deliberately no fallback: if the library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import _build

c_ctx = C.c_void_p
P = C.c_void_p  # every array argument is passed as a raw address
I = C.c_int
D = C.c_double

# name -> (restype, argtypes); must list every function include/sosfront.h declares (tests check this)
PROTOTYPES = {
    "sos_abi_version": (I, []),
    "sos_last_error": (C.c_char_p, []),
    "sos_device_count": (I, [C.POINTER(I)]),
    "sos_ctx_create": (I, [I, C.POINTER(c_ctx)]),
    "sos_ctx_destroy": (I, [c_ctx]),
    "sos_ctx_set_stream": (I, [c_ctx, P]),
    "sos_ctx_get_stream": (P, [c_ctx]),
    "sos_ctx_sync": (I, [c_ctx]),
    "sos_ctx_reserve": (I, [c_ctx, C.c_size_t]),
    "sos_ctx_launch_count": (C.c_int64, [c_ctx]),
    "sos_malloc": (I, [c_ctx, C.c_size_t, C.POINTER(P)]),
    "sos_free": (I, [c_ctx, P]),
    "sos_malloc_host": (I, [C.c_size_t, C.POINTER(P)]),
    "sos_free_host": (I, [P]),
    "sos_memcpy_h2d": (I, [c_ctx, P, P, C.c_size_t]),
    "sos_memcpy_d2h": (I, [c_ctx, P, P, C.c_size_t]),
    "sos_memset": (I, [c_ctx, P, I, C.c_size_t]),
    "sos_lut_pack_f32": (I, [c_ctx, P, P, I, I, P, I, I, P]),
    "sos_lut_pack_f64": (I, [c_ctx, P, P, I, I, P, I, I, P]),
    "sos_remap_u8": (I, [c_ctx, P, I, I, I, I, P, I, I, I, P, P, P]),
    "sos_gum_project": (I, [c_ctx, P, P, I, P]),
    "sos_lut_build": (I, [c_ctx, P, I, I, D, D, D, D, P, P]),
    "sos_hamming_top2": (I, [c_ctx, P, P, P, P, P, P, I, I, I, P, P, P, P]),
    "sos_l2_top2": (I, [c_ctx, P, P, I, P, P, P, P, I, I, I, P, P, P, P, P]),
    "sos_l2f_top2": (I, [c_ctx, P, P, I, P, P, P, P, I, I, I, P, P, P, P, P, P]),
    "sos_hamming_radius": (I, [c_ctx, P, I, P, I, I, P, P, P, P]),
    "sos_match_select": (I, [c_ctx, I, D, P, P, P, P, P, P, P, I, P, P, D, D, P, P, P, P]),
    "sos_lift_pano": (I, [c_ctx, P, P, I, P, P, P]),
    "sos_lift_pano_f64": (I, [c_ctx, P, P, I, P, P, P]),
    "sos_angles_to_sphere_f64": (I, [c_ctx, P, P, I, P]),
    "sos_range_gate_f64": (I, [c_ctx, P, I, D, D, I, P]),
    "sos_triangulate_midpoint_f64": (I, [c_ctx, P, P, P, P, I, P, P, D, D, I, P, P]),
    "sos_lift_gum": (I, [c_ctx, P, P, I, P, P, P]),
    "sos_triangulate_midpoint": (I, [c_ctx, P, P, P, P, I, P, P, D, D, I, P, P]),
    "sos_stereo_lift_triangulate": (I, [c_ctx, P, P, P, P, P, P, P, P, I, I, I, I, P, P, D, D, I, I, P, P, P, P, P, P, P, P]),
    "sos_rgbd_depth_to_z": (I, [c_ctx, P, P, I, I, I, P]),
    "sos_rgbd_backproject": (I, [c_ctx, P, P, I, I, I, P, P, I, D, D, P, P, P]),
    "sos_arun_batch": (I, [c_ctx, P, P, I, I, I, P, P]),
    "sos_pixel_gate": (I, [c_ctx, P, P, I, D, D, P]),
    "sos_ransac_p3d": (I, [c_ctx, P, P, P, P, P, I, I, P, I, P, I, I, I, D, P, P, P, P, P, P]),
    "sos_ransac_score_probe": (I, [c_ctx, P, P, P, P, P, I, I, P, I, P, I, I, D, P, P, P, P, P, P]),
    "sos_ransac_p3p": (I, [c_ctx, P, P, P, P, I, I, P, I, P, I, I, D, P, P, P, P, P, P]),
    "sos_ransac_p3d_eval": (I, [c_ctx, P, P, P, P, P, I, I, P, I, P, I, D, P, P, P]),
    "sos_refit_inliers": (I, [c_ctx, P, P, P, P, I, I, P, P]),
    "sos_median_blur_11": (I, [c_ctx, P, I, I, I, I, P]),
    "sos_median_blur_11_gray": (I, [c_ctx, P, I, I, I, P, P]),
    "sos_bgr_to_gray": (I, [c_ctx, P, C.c_size_t, P]),
    "sos_orb_blur": (I, [c_ctx, P, I, I, I, P]),
    "sos_orb_describe": (I, [c_ctx, P, I, I, I, P, P, P, I, P, P]),
    "sos_corner_min_eigenval": (I, [c_ctx, P, I, I, I, P]),
    "sos_gft_detect": (I, [c_ctx, P, P, I, I, I, I, I, D, D, P, P, P]),
    "sos_dense_triangulate": (I, [c_ctx, P, P, P, I, I, I, D, D, D, I, I, P, P, P, P]),
    "sos_refine_pose": (I, [c_ctx, P, P, P, P, P, I, I, P, I, P, I, I, P, P, P]),
    "sos_ctx_profile_begin": (I, [c_ctx]),
    "sos_ctx_profile_end": (I, [c_ctx, C.c_char_p, C.c_size_t, P, I, C.POINTER(I)]),
    "sos_frontend_profile_begin": (I, [C.c_void_p]),
    "sos_frontend_profile_end": (I, [C.c_void_p, C.c_char_p, C.c_size_t, P, I, C.POINTER(I)]),
    "sos_frontend_create": (I, [c_ctx, P, P, P, C.POINTER(C.c_void_p)]),
    "sos_frontend_destroy": (I, [C.c_void_p]),
    "sos_frontend_reset": (I, [C.c_void_p]),
    "sos_frontend_set_graph": (I, [C.c_void_p, I]),
    "sos_frontend_get_buffers": (I, [C.c_void_p, P]),
    "sos_frontend_set_ref_slots": (I, [C.c_void_p, P]),
    "sos_frontend_promote": (I, [C.c_void_p, I]),
    "sos_frontend_retrack": (I, [C.c_void_p]),
    "sos_frontend_step": (I, [C.c_void_p, P, P, P, P, P, P, P]),
    "sos_frontend_submit_host": (I, [C.c_void_p, P, P, P, P, P, P, P, C.POINTER(I)]),
    "sos_frontend_wait_host": (I, [C.c_void_p, I, P, P]),
    "sos_frontend_host_bytes": (I, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "sos_frontend_step_host": (I, [C.c_void_p, P, P, P, P, P, P, P, P, P]),
    "sos_peak_popc": (I, [c_ctx, C.POINTER(D)]),
    "sos_peak_ffma": (I, [c_ctx, C.POINTER(D)]),
    "sos_peak_dfma": (I, [c_ctx, C.POINTER(D)]),
    "sos_peak_ffma2": (I, [c_ctx, C.POINTER(D)]),
    "sos_peak_tmem_read": (I, [c_ctx, C.POINTER(D)]),
}


class SosError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libsosfront error {code}: {message}")
        self.code = code


_lib = None


def library_path() -> Path:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Load libsosfront.so (built by `python -m vo_single_camera_sos_b200._build` / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not path.exists():
        raise ImportError(
            f"{path} is missing: build it with `python -m vo_single_camera_sos_b200._build` "
            "(there is no CPU fallback for the SOS front-end kernels)")
    lib = C.CDLL(str(path))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.sos_abi_version() != 1:
        raise ImportError(f"{path}: ABI version {lib.sos_abi_version()} != 1; rebuild the library")
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise SosError(code, load().sos_last_error().decode("utf-8", "replace"))
