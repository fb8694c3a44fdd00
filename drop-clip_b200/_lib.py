"""ctypes binding of libdropclip.so (the C ABI declared in include/dropclip.h).

There is no fallback: if the library is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p, POINTER

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DROPCLIP_LIB") or os.path.join(HERE, "libdropclip.so")  # DROPCLIP_LIB: an experimental build

DC_F16, DC_F32, DC_U8, DC_I32, DC_I64, DC_F64 = 0, 1, 2, 3, 4, 5
DC_SIM_NONE, DC_SIM_MAX, DC_SIM_MEAN = 0, 1, 2
DC_GROUND_RAW, DC_GROUND_PAIRED, DC_GROUND_ARGMAX, DC_GROUND_CLASS = 0, 1, 2, 3
ABI_VERSION = 2

P = c_void_p
# name -> (restype, argtypes); must list every DC_API symbol of include/dropclip.h
SIGNATURES = {
    "dc_abi_version": (c_int, []),
    "dc_last_error": (c_char_p, []),
    "dc_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_size_t)]),
    "dc_set_stream_overlap": (c_int, [c_int]),
    "dc_project_visibility": (c_int, [P, P, P, P, P, P, P, c_int, c_int64, c_int, c_int, c_int, c_double, P, c_int, P, P,
                                      c_int, P, P]),
    "dc_visibility_sorted_workspace": (c_size_t, [c_int64, c_int, c_int]),
    "dc_visibility_sorted_groups": (c_int, [c_int, c_int64, c_int]),
    "dc_project_visibility_sorted": (c_int, [P, P, P, P, P, P, c_int, c_int64, c_int64, c_int, c_int, c_int, c_double, P, P, P,
                                             P, c_size_t, P]),
    "dc_unpack_visibility": (c_int, [P, P, P, P, P, c_int, c_int64, c_int64, P, c_int, P]),
    "dc_unpack_visibility_compact": (c_int, [P, P, P, P, P, P, P, P, c_int, c_int64, c_int64, P, c_int, P, c_size_t, P]),
    "dc_unpack_compact_workspace": (c_size_t, [c_int64, c_int]),
    "dc_seg_histogram": (c_int, [P, c_int, c_int64, c_int64, c_int, P, P, P]),
    "dc_view_table": (c_int, [P, P, P, P, P, P, P, c_int64, c_int64, c_int64, c_int, P, P, P, P]),
    "dc_view_score_ld": (c_int, [c_int]),
    "dc_view_score_workspace": (c_size_t, [c_int64, c_int64, c_int, c_int]),
    "dc_view_score": (c_int, [P, c_int, c_int64, c_int, P, P, P, P, c_int64, c_int, c_int, P, c_int, P, c_size_t, P]),
    "dc_view_weights_scratch": (c_size_t, [c_int64, c_int64]),
    "dc_view_weights": (c_int, [P, c_int, P, P, P, P, P, P, P, c_int, c_int64, c_int, c_int, P, P, c_int, c_int, P, c_int64, P, P,
                                ctypes.c_float, P]),
    "dc_segmented_wmean": (c_int, [P, c_int, c_int, P, P, P, P, P, c_int, c_int, P, P]),
    "dc_scatter_to_points": (c_int, [P, P, P, P, c_int, c_int64, c_int, c_int, P, P]),
    "dc_compact_workspace": (c_size_t, [c_int64]),
    "dc_compact_scan": (c_int, [P, c_int64, P, c_int, P, P, P, c_size_t, P]),
    "dc_compact_mask_offsets": (c_int, [P, P, c_int, P, P]),
    "dc_compact_rows": (c_int, [P, c_int64, P, P, c_int64, P, P]),
    "dc_compact_mask": (c_int, [P, c_int, P, P, P, P, P, P, P, c_int, c_int64, c_int, P, P]),
    "dc_pixel_fuse": (c_int, [P, P, P, P, P, P, P, P, c_int, P, c_int, c_int, c_int, P, P, c_int, c_int, c_int, c_int64,
                              c_int, c_int, c_int, P, P, P, c_int, c_int64, c_int, P, c_size_t, P]),
    "dc_pixel_fuse_mma_workspace": (c_size_t, [c_int64, c_int64, c_int, c_int, c_int, c_int]),
    "dc_pixel_fuse_mma": (c_int, [P, P, P, P, P, P, P, P, c_int, P, c_int, c_int, c_int, P, P, c_int, c_int, c_int, c_int64,
                                  c_int, c_int, c_int, P, P, P, c_int, c_int64, c_int64, c_int64, c_int, P, c_size_t, P]),
    "dc_pixel_fuse_workspace": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "dc_spatial_sort_workspace": (c_size_t, [c_int]),
    "dc_spatial_sort": (c_int, [P, P, c_int, c_int64, c_int64, P, P, P, c_size_t, P]),
    "dc_pixel_normalize": (c_int, [P, P, P, P, P, P, c_int, c_int64, c_int, P]),
    "dc_view_clip_gather": (c_int, [P, c_int64, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P, P]),
    "dc_voxelize_workspace": (c_size_t, [c_int64]),
    "dc_voxelize": (c_int, [P, P, c_int, c_int64, c_float, P, ctypes.c_int32, P, P, P, P, P, P, c_size_t, P]),
    "dc_voxel_gather": (c_int, [P, c_int64, P, P, P, c_int, c_int64, P, P]),
    "dc_row_normalize": (c_int, [P, c_int, c_int64, c_int, c_int, P, P, P]),
    "dc_ground_init_minmax": (c_int, [P, P]),
    "dc_ground_workspace": (c_size_t, [c_int64, c_int, c_int]),
    "dc_ground": (c_int, [P, P, c_int64, P, P, c_int, c_int, c_int, c_float, c_int, P, c_int, P, P, P, P, c_size_t, P]),
    "dc_predict_workspace": (c_size_t, [c_int64, c_int, c_int, c_int, c_int, c_int]),
    "dc_predict": (c_int, [P, c_int, c_int64, P, c_int, c_int, c_int, c_int, c_float, c_int, c_float, P, P, P, P, c_size_t, P]),
    "dc_predict_queries_workspace": (c_size_t, [c_int64, c_int, c_int, c_int64, c_int, c_int, c_int]),
    "dc_predict_queries": (c_int, [P, c_int, c_int64, P, c_int, c_int, c_int, P, P, P, c_int, c_int, c_float, c_int, c_float, P,
                                   P, P, c_size_t, P]),
    "dc_predict_many_workspace": (c_size_t, [c_int, P, P, P, c_int64, c_int, c_int, c_int]),
    "dc_predict_many": (c_int, [P, c_int, P, c_int, c_int, c_int, P, P, P, P, P, P, c_int, c_float, c_int, c_float, P, P, P,
                                c_size_t, P]),
    "dc_minmax_threshold": (c_int, [P, c_int64, P, c_int, c_float, c_int, P, P]),
    "dc_backproject": (c_int, [P, c_int, c_int, c_int, P, c_int, c_int, P, P, P]),
    "dc_points_to_pixels": (c_int, [P, c_int64, P, P, P]),
    "dc_transform_points": (c_int, [P, c_int64, P, P, P]),
    "dc_sort_workspace": (c_size_t, [c_int64]),
    "dc_unique_max_pool": (c_int, [P, P, c_int, c_int, c_int64, P, P, P, P, c_size_t, P]),
    "dc_voxel_down_mean": (c_int, [P, c_int64, c_double, P, P, P, P, c_size_t, P]),
    "dc_voxel_down_trace": (c_int, [P, P, P, c_int64, c_double, P, P, P, P, P, P, P, c_size_t, P]),
    "dc_nearest_index": (c_int, [P, c_int64, P, c_int64, P, P, P]),
    "dc_binary_iou_counts": (c_int, [P, P, c_int, P, c_int, c_int64, c_float, c_int, c_int, P, P, P]),
    "dc_class_iou_workspace": (c_size_t, [c_int]),
    "dc_class_iou_hist": (c_int, [P, P, c_int, c_int64, c_int, c_int64, P, P, P, P, c_size_t, P]),
    "dc_sample_keep_flags": (c_int, [P, P, P, P, P, c_int, c_int64, P, P]),
    "dc_sample_gather": (c_int, [P, P, P, P, P, P, P, P, P, P, P, c_int, c_int64, c_int64, c_int64, c_int, c_int, P, P, P, P,
                                 P, P, P, P, P]),
    "dc_host_gather_copy": (c_int, [P, c_int64, c_int64, P, c_int]),
    "dc_host_gather_narrow_i64_u8": (c_int, [P, c_int64, c_int64, P, c_int, POINTER(c_int)]),
}

_lib = None


class DropClipError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"libdropclip error {status}: {message}")
        self.status = status


def load(path: str = LIB_PATH):
    """Loads the shared library and binds every declared symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `python -m dropclip_b200.build` (or __graft_entry__.build()). "
            "There is no CPU fallback.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.dc_abi_version() != ABI_VERSION:
        raise ImportError(f"libdropclip ABI {lib.dc_abi_version()} != expected {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise DropClipError(rc, (load().dc_last_error() or b"").decode())


def ptr(t):
    """Device (or None) pointer of a torch tensor."""
    return None if t is None else c_void_p(t.data_ptr())


def current_stream():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def torch_dtype_code(dtype) -> int:
    import torch
    return {torch.float16: DC_F16, torch.float32: DC_F32, torch.uint8: DC_U8, torch.int32: DC_I32,
            torch.int64: DC_I64, torch.float64: DC_F64}[dtype]
