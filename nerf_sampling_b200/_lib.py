"""ctypes binding of ``libb200nerf.so`` (the C ABI declared in ``include/b200nerf.h``).

There is no fallback: if the library is missing, stale or fails to load, every operator raises.
"""

from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import _build

_LIB: Optional[C.CDLL] = None

P = C.c_void_p
I = C.c_int
F = C.c_float
SZ = C.c_size_t

# name -> (restype, argtypes); mirrors include/b200nerf.h one to one
SIGNATURES = {
    "b200nerf_version": (I, []),
    "b200nerf_last_error": (C.c_char_p, []),
    "b200nerf_launch_count": (C.c_ulonglong, []),
    "b200nerf_nerf_wpack_bytes": (SZ, [I]),
    "b200nerf_nerf_aux_floats": (SZ, []),
    "b200nerf_nerf_pack": (I, [P, I, P, P]),
    "b200nerf_nerf_pack_multires": (I, [P, I, I, I, P, P]),
    "b200nerf_depthnet_wpack_bytes": (SZ, [I, I]),
    "b200nerf_depthnet_aux_floats": (SZ, [I]),
    "b200nerf_depthnet_pack": (I, [P, P, P, I, P, P, I, P, P]),
    "b200nerf_depthnet_pack_multires": (I, [P, P, P, I, P, P, I, I, P, P]),
    "b200nerf_get_rays": (I, [I, I, F, F, F, F, P, P, P, P, P]),
    "b200nerf_get_rays_at": (I, [I, I, F, F, F, F, P, P, I, P, P, P, P]),
    "b200nerf_gather_pixels": (I, [P, P, I, I, P, P]),
    "b200nerf_normalize_dirs": (I, [P, I, P, P]),
    "b200nerf_depthnet_fwd": (I, [P, P, I, I, P, P, I, F, F, F, P, P]),
    "b200nerf_place_samples": (I, [P, P, I, I, I, F, F, P, P]),
    "b200nerf_points": (I, [P, P, P, I, I, P, P]),
    "b200nerf_nerf_mlp_fwd": (I, [P, P, I, P, P, P, P, P, I, I, P, P]),
    "b200nerf_nerf_fast_wpack_bytes": (SZ, []),
    "b200nerf_nerf_pack_fast": (I, [P, I, P]),
    "b200nerf_nerf_pack_fast_multires": (I, [P, I, I, I, P]),
    "b200nerf_nerf_mlp_fast_fwd": (I, [P, P, I, P, P, P, P, P, I, I, P, P, P, I, F, P]),
    "b200nerf_nerf_mlp_guarded_fwd": (I, [P, P, P, I, P, P, P, P, P, I, I, F, P, P, P]),
    "b200nerf_composite_fwd": (I, [P, P, P, P, I, I, I, P, P, P, P, P, P, P]),
    "b200nerf_composite_tile_fwd": (I, [P, P, P, P, I, I, I, P, P, P, P, P, P]),
    "b200nerf_composite_bwd": (I, [P, P, P, P, I, I, I, P, P, P, P, P, P, P, P, P]),
    "b200nerf_place_samples_bwd": (I, [P, P, I, I, I, F, F, P, P, P]),
    "b200nerf_points_bwd": (I, [P, P, I, I, P, P]),
    "b200nerf_render_depthnet_tile": (I, [P, P, I, I, P, P, P, P, I, I, I, P, F, F, F, P, P, P, P, P, P, P, P, P]),
    "b200nerf_set_sm_limit": (I, [I]),
    "b200nerf_nerf_query": (I, [P, P, P, P, P, P, I, I, P, P, P]),
    "b200nerf_render_depthnet": (I, [P, P, I, I, P, P, P, P, I, I, I, P, F, F, F, P, P, P, P, P, P, P, P, P, P]),
    "b200nerf_render_host_ws_bytes": (SZ, [I, I]),
    "b200nerf_render_depthnet_host": (I, [P, P, I, I, P, P, P, I, I, I, P, F, F, F, P, P, P, P]),
    "b200nerf_coarse_depths": (I, [P, P, P, I, I, I, P, P, P]),
    "b200nerf_sample_pdf": (I, [P, P, P, I, I, I, I, P, P, P]),
    "b200nerf_sample_pdf_merge": (I, [P, P, P, I, I, I, I, P, P, P, P]),
    "b200nerf_argmax_gather": (I, [P, P, P, I, I, P, P, P, P, P]),
    "b200nerf_umma_selftest": (I, [P, P, P, I, I, P]),
    "b200nerf_debug_set_tgemm_timeline": (None, [P]),
    "b200nerf_debug_sgemm": (I, [I, I, I, P, C.c_long, C.c_long, P, C.c_long, C.c_long, P, I, I, P, I, F, I, P]),
    "b200nerf_debug_depthnet_train_route": (I, [P, I, P, I, P, I]),
    "b200nerf_debug_depthnet_train_route_multires": (I, [P, I, P, I, P, I, I]),
    "b200nerf_depthnet_train_ws_floats": (SZ, [I, I, P, I, P]),
    "b200nerf_depthnet_train_ws_floats_multires": (SZ, [I, I, P, I, P, I]),
    "b200nerf_depthnet_n_params": (I, [I, I]),
    "b200nerf_depthnet_train_fwd": (I, [P, I, P, I, P, P, P, I, F, F, F, P, P, P]),
    "b200nerf_depthnet_train_fwd_multires": (I, [P, I, P, I, P, I, P, P, I, F, F, F, P, P, P]),
    "b200nerf_depthnet_train_bwd": (I, [P, I, P, I, P, I, F, F, P, P, P, P]),
    "b200nerf_depthnet_train_bwd_multires": (I, [P, I, P, I, P, I, I, F, F, P, P, P, P]),
    "b200nerf_depthnet_train_jac": (I, [P, I, P, I, P, I, F, F, P, P, P]),
    "b200nerf_depthnet_train_jac_multires": (I, [P, I, P, I, P, I, I, F, F, P, P, P]),
    "b200nerf_depthnet_train_bwd_jac": (I, [P, I, P, I, P, I, F, F, P, P, P, P, P]),
    "b200nerf_depthnet_train_bwd_jac_multires": (I, [P, I, P, I, P, I, I, F, F, P, P, P, P, P]),
    "b200nerf_nerf_point_ws_floats": (SZ, [I]),
    "b200nerf_nerf_point_jvp": (I, [P, P, P, P, P, I, P, P, P, P]),
    "b200nerf_nerf_point_ws_floats_multires": (SZ, [I, I, I]),
    "b200nerf_nerf_point_jvp_multires": (I, [P, I, I, P, P, P, P, I, P, P, P, P]),
    "b200nerf_nerf_point_jvp_packed_ws_bytes": (SZ, [I]),
    "b200nerf_nerf_point_jvp_packed": (I, [P, P, P, P, P, P, I, P, P, P, P]),
    "b200nerf_nerf_samples_ws_floats_multires": (SZ, [I, I, I, I]),
    "b200nerf_nerf_samples_jvp_multires": (I, [P, I, I, P, P, P, P, I, I, P, P, P, P]),
    "b200nerf_nerf_samples_jvp_packed_ws_bytes": (SZ, [I, I]),
    "b200nerf_nerf_samples_jvp_packed": (I, [P, P, P, P, P, P, I, I, P, P, P, P]),
    "b200nerf_nerf_pts_jvp_packed": (I, [P, P, P, P, I, I, P, P, P, P]),
    "b200nerf_debug_catchain_img_bytes": (SZ, [I]),
    "b200nerf_debug_catchain_pack": (I, [P, P, P, P, I, P, P, P, P]),
    "b200nerf_train_loss": (I, [P, P, P, P, P, I, P, P, P, P]),
    "b200nerf_adam_step": (I, [P, P, P, P, SZ, F, F, F, F, I, F, P]),
    "b200nerf_adam_step_multi": (I, [P, I, F, F, F, F, I, F, P]),
    "b200nerf_adam_step_multi_dev": (I, [P, I, P, P, P]),
}


class NerfModel(C.Structure):
    """``b200nerf_nerf_model`` of include/b200nerf.h."""

    _fields_ = [("wpack", P), ("wpack_fast", P), ("aux", P), ("prec", I), ("guard_kappa", F)]


class B200NerfError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the library; raises if it cannot be loaded."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = _build.LIB_PATH
    if not os.path.exists(path):
        raise B200NerfError(
            f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU or eager fallback."
        )
    handle = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if handle.b200nerf_version() != 100:
        raise B200NerfError("libb200nerf.so version mismatch; rebuild")
    _LIB = handle
    return handle


def check(rc: int) -> None:
    if rc != 0:
        raise B200NerfError(lib().b200nerf_last_error().decode())


def launch_count() -> int:
    return int(lib().b200nerf_launch_count())
