"""ctypes binding of libhands_b200.so (the C ABI declared in include/hands_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc; if that fails, or a
call returns non-zero, a RuntimeError is raised.
"""
import ctypes
import os

from . import _build

c_float_p = ctypes.c_void_p  # device / host pointers are passed as integers
_lib = None

SYMBOLS = {
    "hb_last_error_string": (ctypes.c_char_p, []),
    "hb_version": (ctypes.c_int, []),
    "hb_launch_count": (ctypes.c_uint64, []),
    "hb_mano_create": (ctypes.c_int, [ctypes.c_void_p] * 8 + [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "hb_mano_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "hb_mano_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "hb_mano_head_fwd": (
        ctypes.c_int,
        [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
         ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_float]
        + [ctypes.c_void_p] * 6 + [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p],
    ),
    "hb_mano_head_bwd": (
        ctypes.c_int,
        [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
         ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_float]
        + [ctypes.c_void_p] * 6 + [ctypes.c_void_p] * 5 + [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p],
    ),
    "hb_mano_head_bwd_reuse": (
        ctypes.c_int,
        [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
         ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_float]
        + [ctypes.c_void_p] * 6 + [ctypes.c_void_p] * 5 + [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p],
    ),
    "hb_matrix_to_axis_angle_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_matrix_to_axis_angle_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_rot6d_to_rotmat_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_rot6d_to_rotmat_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_project2d_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_project2d_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_weak_to_persp_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_weak_to_persp_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_persp_to_weak_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_rot_apply": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_kp_loss_fwd": (ctypes.c_int, [ctypes.c_void_p] * 8 + [ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_kp_loss_bwd": (ctypes.c_int, [ctypes.c_void_p] * 7 + [ctypes.c_int] + [ctypes.c_void_p] * 5),
    "hb_vec_loss_fwd": (ctypes.c_int, [ctypes.c_void_p] * 8 + [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_vec_loss_bwd": (ctypes.c_int, [ctypes.c_void_p] * 8 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 5),
    "hb_axis_angle_to_matrix": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_mrrpe": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_procrustes_metrics": (ctypes.c_int, [ctypes.c_void_p] * 2 + [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 8),
    "hb_gt_process": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_float] + [ctypes.c_void_p] * 4),
    "hb_kpe_features": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 5),
    "hb_pcl_setup": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_pcl_homography_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_pcl_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_pcl_set_exact": (ctypes.c_int, [ctypes.c_int]),
    "hb_pcl_fwd_u8": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_pcl_bwd_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "hb_pcl_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "hb_pcl_bwd_stages": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]),
    "hb_pcl_fwd_bf16": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_pcl_fwd_u8_bf16": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_pcl_bwd_bf16": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "hb_sil_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "hb_sil_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "hb_sil_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "hb_sil_fwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_float,
                                  ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "hb_sil_bwd": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                  ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_mask_l1_loss_fwd": (ctypes.c_int, [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "hb_mask_l1_loss_bwd": (ctypes.c_int, [ctypes.c_void_p] * 5 + [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
}

PCL_PARAM_FLOATS = 32
KP_SUMS = 8
POSE_AXIS_ANGLE, POSE_ROTMAT, POSE_ROT6D = 0, 1, 2
ROT6D_ROWS, ROT6D_COLS, ROT6D_COLS_PAIRED = 0, 1, 2
ROT6D_LAYOUTS = {"rows": ROT6D_ROWS, "cols": ROT6D_COLS, "cols_paired": ROT6D_COLS_PAIRED}


def lib_path():
    return _build.LIB


def load():
    """Load (building first if needed) and type the library.  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build()   # no-op when the binary's source digest matches the tree; rebuilds a stale or missing one
    lib = ctypes.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here means the .so does not match include/hands_b200.h
        fn.restype = res
        fn.argtypes = args
    if lib.hb_version() != _build.header_version():
        raise RuntimeError(f"libhands_b200.so reports version {lib.hb_version()}, include/hands_b200.h declares {_build.header_version()}")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().hb_last_error_string()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def launch_count():
    return int(load().hb_launch_count())
