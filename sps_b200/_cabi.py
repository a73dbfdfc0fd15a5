"""ctypes binding of ``include/sps_b200.h`` -- the only way host code reaches the kernels.

There is deliberately no fallback: if ``libsps_b200.so`` cannot be loaded the import of the
product path raises (the CUDA extension IS the product)."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SPS_B200_LIB: an alternative build of the same library (kernel A/B measurements, tools/build_variant.py)
LIB_PATH = os.environ.get("SPS_B200_LIB") or os.path.join(HERE, "libsps_b200.so")

SPS_OK, SPS_ERR_BAD_ARG, SPS_ERR_CAPACITY, SPS_ERR_COORD_RANGE, SPS_ERR_CUDA, SPS_ERR_UNSUPPORTED, SPS_ERR_STATE = range(7)
SPS_NUM_LEVELS = 5
SPS_CONV_NBR, SPS_CONV_UP = 0, 1
SPS_BACKEND_AUTO, SPS_BACKEND_FP32, SPS_BACKEND_TF32, SPS_BACKEND_F16 = 0, 1, 2, 3
SPS_IO_F32, SPS_IO_F16 = 0, 1
SPS_CONV_FOLD_LO, SPS_CONV_OUT_SPLIT, SPS_CONV_MAP_PARENT = 1, 2, 4
SPS_PACK_IN_SPLIT, SPS_PACK_IN2_SPLIT, SPS_PACK_FOLD_LO = 1, 2, 4
_ERR_NAMES = {1: "SPS_ERR_BAD_ARG", 2: "SPS_ERR_CAPACITY", 3: "SPS_ERR_COORD_RANGE", 4: "SPS_ERR_CUDA",
              5: "SPS_ERR_UNSUPPORTED", 6: "SPS_ERR_STATE"}

# every symbol include/sps_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "sps_version", "sps_last_error", "sps_workspace_bytes", "sps_ctx_create", "sps_ctx_destroy", "sps_ctx_status",
    "sps_ctx_level", "sps_ctx_inverse_map", "sps_voxelize", "sps_build_maps", "sps_unpack_coords", "sps_conv_fwd",
    "sps_net_create", "sps_net_destroy", "sps_net_set_tensor", "sps_net_set_output", "sps_net_device_bytes", "sps_net_finalize",
    "sps_forward", "sps_forward_features", "sps_forward_host", "sps_unet_forward", "sps_devox_sigmoid", "sps_ctx_launch_count",
    "sps_map_bytes", "sps_map_build", "sps_map_destroy", "sps_submap_crop_voxel", "sps_submap_crop_radius",
    "sps_assemble", "sps_memcpy_d2h", "sps_memcpy_h2d", "sps_infer_scan", "sps_infer_scan_scratch_bytes", "sps_conv_kmajor_ld", "sps_conv_pack_kmajor", "sps_conv_kmajor_ld_f16", "sps_conv_pack_kmajor_f16", "sps_conv_kmajor_ld_f16x", "sps_conv_pack_kmajor_f16x", "sps_conv_kmajor_ld_f16s", "sps_conv_pack_kmajor_f16s", "sps_kernel_map_tile_masks", "sps_tma_weights_available", "sps_ctx_set_pattern_sort",
    "sps_ctx_set_conv_backend", "sps_profile_enable", "sps_profile_read", "sps_ctx_pair_count",
    "sps_confusion_counts", "sps_voxel_mean", "sps_voxel_sum", "sps_gather_rows", "sps_affine_relu",
    "sps_pointcloud2_unpack", "sps_transform_points", "sps_pointcloud2_pack_scratch_bytes", "sps_pointcloud2_pack",
    "sps_ballmap_bytes", "sps_ballmap_build", "sps_ballmap_destroy", "sps_ball_query_scratch_bytes", "sps_submap_ball_query",
    "sps_radius_batch_scratch_bytes", "sps_radius_batch", "sps_predict_radius_batch",
    "sps_prune_batch_scratch_bytes", "sps_prune_batch", "sps_infer_prune_batch",
    "sps_filter_scans_batch_scratch_bytes", "sps_filter_scans_batch", "sps_gather_segments",
]


class LevelView(C.Structure):
    _fields_ = [("keys", C.c_void_p), ("count", C.c_void_p), ("nbr3", C.c_void_p), ("nbr5", C.c_void_p),
                ("parent", C.c_void_p), ("child", C.c_void_p), ("ld", C.c_int64),
                ("perm", C.c_void_p), ("tile_mask", C.c_void_p), ("tile_slices", C.c_void_p)]


class ConvArgs(C.Structure):
    _fields_ = [("mode", C.c_int), ("K", C.c_int), ("cin", C.c_int), ("cout", C.c_int),
                ("map", C.c_void_p), ("map_ld", C.c_int64), ("n_out", C.c_void_p), ("n_out_max", C.c_int64),
                ("in_", C.c_void_p), ("in_ld", C.c_int64), ("weight", C.c_void_p), ("shift", C.c_void_p),
                ("in2", C.c_void_p), ("in2_ld", C.c_int64), ("cin2", C.c_int), ("weight2", C.c_void_p),
                ("res", C.c_void_p), ("res_ld", C.c_int64), ("relu", C.c_int),
                ("out", C.c_void_p), ("out_ld", C.c_int64),
                ("head_w", C.c_void_p), ("head_b", C.c_float), ("head_out", C.c_void_p),
                ("weight_kmajor", C.c_void_p), ("kmajor_ld", C.c_int64), ("round_out", C.c_int),
                ("tile_mask", C.c_void_p), ("perm", C.c_void_p), ("tile_slices", C.c_void_p), ("io_dtype", C.c_int),
                ("backend", C.c_int), ("flags", C.c_int), ("cin_split", C.c_int)]


class SpsError(RuntimeError):
    def __init__(self, code, where, detail=""):
        self.code = code
        super().__init__(f"{where} failed: {_ERR_NAMES.get(code, code)}{(' -- ' + detail) if detail else ''}")


_lib = None


def load() -> C.CDLL:
    """Load the in-tree shared library; build it first when it is missing and nvcc exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build  # raises if nvcc is absent: no silent fallback
        _build.build()
    lib = C.CDLL(LIB_PATH)
    vp, i64, i32, f32, sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t
    sig = {
        "sps_version": (C.c_char_p, []),
        "sps_last_error": (C.c_char_p, []),
        "sps_workspace_bytes": (sz, [i64]),
        "sps_net_set_output": (i32, [vp, i32, i32]),
        "sps_forward_features": (i32, [vp, vp, vp, i64, i64, vp, f32, vp, vp]),
        "sps_ctx_create": (i32, [C.POINTER(vp), vp, sz, i64]),
        "sps_ctx_destroy": (i32, [vp]),
        "sps_ctx_status": (i32, [vp, vp]),
        "sps_ctx_level": (i32, [vp, i32, C.POINTER(LevelView)]),
        "sps_ctx_inverse_map": (vp, [vp]),
        "sps_voxelize": (i32, [vp, vp, i64, i64, f32, vp]),
        "sps_build_maps": (i32, [vp, vp]),
        "sps_unpack_coords": (i32, [vp, i32, vp, vp]),
        "sps_conv_fwd": (i32, [C.POINTER(ConvArgs), vp]),
        "sps_net_create": (i32, [C.POINTER(vp)]),
        "sps_net_destroy": (i32, [vp]),
        "sps_net_set_tensor": (i32, [vp, C.c_char_p, vp, i64]),
        "sps_net_device_bytes": (sz, []),
        "sps_net_finalize": (i32, [vp, vp, sz, vp]),
        "sps_forward": (i32, [vp, vp, vp, i64, i64, f32, vp, vp]),
        "sps_forward_host": (i32, [vp, vp, vp, i64, i64, f32, vp, vp]),
        "sps_unet_forward": (i32, [vp, vp, vp, vp, vp]),
        "sps_devox_sigmoid": (i32, [vp, vp, i64, vp, vp]),
        "sps_ctx_launch_count": (i32, [vp]),
        "sps_map_bytes": (sz, [i64]),
        "sps_map_build": (i32, [C.POINTER(vp), vp, sz, vp, i64, f32, vp]),
        "sps_map_destroy": (i32, [vp]),
        "sps_submap_crop_voxel": (i32, [vp, vp, i64, vp, sz, vp, vp, vp]),
        "sps_submap_crop_radius": (i32, [vp, i64, C.POINTER(C.c_double), C.c_double, vp, vp, vp, sz, vp]),
        "sps_assemble": (i32, [vp, i64, vp, vp, i64, f32, vp, vp]),
        "sps_memcpy_d2h": (i32, [vp, vp, sz, vp]),
        "sps_memcpy_h2d": (i32, [vp, vp, sz, vp]),
        "sps_infer_scan": (i32, [vp, vp, vp, vp, i64, f32, vp, vp, sz, vp, vp]),
        "sps_infer_scan_scratch_bytes": (sz, [i64]),
        "sps_ctx_set_pattern_sort": (i32, [vp, i32]),
        "sps_tma_weights_available": (i32, []),
        "sps_kernel_map_tile_masks": (i32, [vp, i64, i32, vp, i64, vp, vp]),
        "sps_conv_kmajor_ld": (i64, [i32, i32, i32]),
        "sps_conv_pack_kmajor": (i32, [vp, i32, i32, i32, vp, i32, vp]),
        "sps_conv_kmajor_ld_f16": (i64, [i32, i32, i32]),
        "sps_conv_pack_kmajor_f16": (i32, [vp, i32, i32, i32, vp, i32, vp]),
        "sps_conv_kmajor_ld_f16x": (i64, [i32, i32, i32, i32]),
        "sps_conv_pack_kmajor_f16x": (i32, [vp, i32, i32, i32, vp, i32, i32, vp]),
        "sps_conv_kmajor_ld_f16s": (i64, [i32, i32, i32, i32, i32]),
        "sps_conv_pack_kmajor_f16s": (i32, [vp, i32, i32, i32, vp, i32, i32, i32, vp]),
        "sps_ctx_set_conv_backend": (i32, [vp, i32]),
        "sps_confusion_counts": (i32, [vp, vp, i64, i64, f32, f32, vp, vp, vp]),
        "sps_voxel_mean": (i32, [vp, vp, i64, i32, vp, vp, vp]),
        "sps_voxel_sum": (i32, [vp, vp, i64, i32, vp, vp, vp]),
        "sps_gather_rows": (i32, [vp, i64, i32, vp, i64, vp, vp]),
        "sps_affine_relu": (i32, [vp, i64, i32, i64, vp, vp, i32, vp, i64, vp]),
        "sps_pointcloud2_unpack": (i32, [vp, i64, i64, i64, i64, i32, vp, vp, i32, vp, vp]),
        "sps_transform_points": (i32, [vp, i64, i64, vp, vp, vp]),
        "sps_pointcloud2_pack_scratch_bytes": (sz, [i64]),
        "sps_pointcloud2_pack": (i32, [vp, i64, i64, vp, f32, vp, vp, vp, sz, vp]),
        "sps_ballmap_bytes": (sz, [i64]),
        "sps_ballmap_build": (i32, [C.POINTER(vp), vp, sz, vp, i64, C.c_double, vp]),
        "sps_ballmap_destroy": (i32, [vp]),
        "sps_ball_query_scratch_bytes": (sz, [i64]),
        "sps_submap_ball_query": (i32, [vp, vp, i64, vp, vp, i64, vp, vp, sz, vp]),
        "sps_radius_batch_scratch_bytes": (sz, [i64, i32]),
        "sps_radius_batch": (i32, [vp, vp, i64, vp, i32, vp, i64, vp, vp, vp, sz, vp]),
        "sps_predict_radius_batch": (i32, [vp, vp, vp, vp, i64, vp, i32, vp, i64, vp, vp, vp, sz, f32, f32, vp, vp, vp,
                                           vp]),
        "sps_prune_batch_scratch_bytes": (sz, [i64, i32]),
        "sps_prune_batch": (i32, [vp, vp, i64, vp, i32, vp, vp, vp, vp, vp, sz, vp]),
        "sps_infer_prune_batch": (i32, [vp, vp, vp, vp, i64, vp, i32, vp, vp, vp, vp, vp, sz, f32, vp, vp]),
        "sps_filter_scans_batch_scratch_bytes": (sz, [i64, i32]),
        "sps_filter_scans_batch": (i32, [vp, vp, vp, vp, i64, vp, i32, vp, f32, f32, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                          vp, sz, vp]),
        "sps_gather_segments": (i32, [vp, i32, i64, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp]),
        "sps_profile_enable": (i32, [vp, i32]),
        "sps_profile_read": (i32, [vp, vp, vp, i32, C.POINTER(i32)]),
        "sps_ctx_pair_count": (i32, [vp, i32, i32, C.POINTER(i64), vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int, where: str):
    if code != SPS_OK:
        detail = load().sps_last_error().decode() if code == SPS_ERR_CUDA else ""
        raise SpsError(code, where, detail)
