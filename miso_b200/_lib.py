"""ctypes binding of libmisob200.so (the C ABI declared in include/misob200.h).

There is no CPU fallback: if the CUDA library is missing or does not load, every operator
raises. `load()` never builds on import; `miso_b200.build.build()` (or
`__graft_entry__.build()`) produces the library in-tree.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

MB_MAX_LEVELS = 8
MB_MAX_ANCHORS_PER_LOC = 16
MB_MAX_IMAGES = 64

MB_OK = 0
MB_ERRORS = {-1: "invalid argument", -2: "workspace too small", -3: "unsupported configuration"}

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmisob200.so")

_p = C.c_void_p
_i64, _i32, _f32, _f64, _sz = C.c_int64, C.c_int32, C.c_float, C.c_double, C.c_size_t


class RoiAlignParams(C.Structure):
    _fields_ = [
        ("num_levels", _i32), ("num_images", _i32), ("channels", _i32),
        ("pooled_h", _i32), ("pooled_w", _i32), ("sampling_ratio", _i32),
        ("aligned", _i32), ("exact", _i32),
        ("height", _i32 * MB_MAX_LEVELS), ("width", _i32 * MB_MAX_LEVELS),
        ("spatial_scale", _f32 * MB_MAX_LEVELS), ("level_thresholds", _f32 * MB_MAX_LEVELS),
        ("features", _p * MB_MAX_LEVELS),
        ("boxes_per_image", _i32), ("box_counts", _p), ("channels_last", _i32), ("force_gather", _i32),
    ]


class RpnParams(C.Structure):
    _fields_ = [
        ("num_images", _i32), ("num_levels", _i32),
        ("feat_h", _i32 * MB_MAX_LEVELS), ("feat_w", _i32 * MB_MAX_LEVELS),
        ("stride_h", _i32 * MB_MAX_LEVELS), ("stride_w", _i32 * MB_MAX_LEVELS),
        ("anchors_per_loc", _i32 * MB_MAX_LEVELS),
        ("base_anchors", ((_f32 * 4) * MB_MAX_ANCHORS_PER_LOC) * MB_MAX_LEVELS),
        ("image_h", _i32 * MB_MAX_IMAGES), ("image_w", _i32 * MB_MAX_IMAGES),
        ("pre_nms_top_n", _i32), ("post_nms_top_n", _i32),
        ("nms_thresh", _f64),
        ("score_thresh", _f32), ("min_size", _f32),
        ("wx", _f32), ("wy", _f32), ("ww", _f32), ("wh", _f32), ("bbox_xform_clip", _f32),
        ("trick_numel", _i64),
        ("objectness", _p * MB_MAX_LEVELS), ("deltas", _p * MB_MAX_LEVELS),
    ]


class DetParams(C.Structure):
    _fields_ = [
        ("num_images", _i32), ("num_classes", _i32), ("max_props_per_image", _i32),
        ("detections_per_img", _i32),
        ("image_h", _i32 * MB_MAX_IMAGES), ("image_w", _i32 * MB_MAX_IMAGES),
        ("orig_h", _i32 * MB_MAX_IMAGES), ("orig_w", _i32 * MB_MAX_IMAGES),
        ("nms_thresh", _f64),
        ("score_thresh", _f32), ("min_size", _f32),
        ("wx", _f32), ("wy", _f32), ("ww", _f32), ("wh", _f32), ("bbox_xform_clip", _f32),
        ("trick_numel", _i64),
    ]


class CropParams(C.Structure):
    _fields_ = [
        ("num_images", _i32), ("capacity", _i32), ("channels", _i32),
        ("image_h", _i32 * MB_MAX_IMAGES), ("image_w", _i32 * MB_MAX_IMAGES),
        ("images", _p * MB_MAX_IMAGES),
        ("threshold", _f32), ("boxes_are_xywh", _i32),
    ]


# symbol -> (restype, argtypes); tests/test_abi.py checks this table against include/misob200.h
class TransformParams(C.Structure):     # mirrors mb_transform_params
    _fields_ = [("num_images", _i32), ("channels", _i32), ("images", C.c_void_p * 64),
                ("in_h", _i32 * 64), ("in_w", _i32 * 64), ("out_h", _i32 * 64), ("out_w", _i32 * 64),
                ("mean", _f32 * 4), ("std", _f32 * 4), ("pad_h", _i32), ("pad_w", _i32)]


SIGNATURES = {
    "mb_abi_version": (C.c_int, []),
    "mb_build_info": (C.c_char_p, []),
    "mb_nms_workspace_bytes": (_sz, [_i64, _i32]),
    "mb_nms": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _f64, _p, _p, _p, _sz, _p, _sz, _p]),
    "mb_roi_align_workspace_bytes": (_sz, [C.POINTER(RoiAlignParams), _i64]),
    "mb_multiscale_roi_align": (C.c_int, [C.POINTER(RoiAlignParams), _p, _i64, _p, _p, _p, _sz, _p]),
    "mb_roi_align_tma_launches": (_i64, []),
    "mb_box_decode": (C.c_int, [_p, _p, _i64, _i32, _f32, _f32, _f32, _f32, _f32, _p, _p]),
    "mb_clip_boxes": (C.c_int, [_p, _i64, _f32, _f32, _p, _p]),
    "mb_box_convert": (C.c_int, [_p, _i64, _i32, _i32, _p, _p]),
    "mb_remove_small": (C.c_int, [_p, _i64, _f32, _p, _p, _p]),
    "mb_resize_boxes": (C.c_int, [_p, _i64, _f32, _f32, _p, _p]),
    "mb_grid_anchors": (C.c_int, [C.POINTER(_f32), _i32, _i32, _i32, _i32, _i32, _p, _p]),
    "mb_rpn_workspace_bytes": (_sz, [C.POINTER(RpnParams)]),
    "mb_rpn_proposals": (C.c_int, [C.POINTER(RpnParams), _p, _p, _p, _p, _p, _sz, _p]),
    "mb_det_workspace_bytes": (_sz, [C.POINTER(DetParams)]),
    "mb_det_postprocess": (C.c_int, [C.POINTER(DetParams), _p, _p, _p, _p, _i32, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "mb_crop_plan": (C.c_int, [C.POINTER(CropParams), _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "mb_crop_gather": (C.c_int, [C.POINTER(CropParams), _p, _p, _p, _p, _p, _i64, _p]),
    "mb_mosaic_pack": (C.c_int, [_p, _p, _p, _p, _p, _i32, _i32, C.c_float, _i64, _p, _p]),
    "mb_mosaic_unpack": (C.c_int, [_p, _i64, _p, _p, _p, _p]),
    "mb_seam_nms_workspace_bytes": (_sz, [_i64, _i32, _i64]),
    "mb_seam_nms": (C.c_int, [_p, _i64, _i32, _f64, _i64, _p, _p, _p, _p, _sz, _p]),
    "mb_seam_select": (C.c_int, [_p, _p, _i64, _i64, _p, _p, _p]),
    "mb_box_iou": (C.c_int, [_p, _i64, _p, _i64, _p, _p]),
    "mb_match_encode_workspace_bytes": (_sz, [_i64, _i64]),
    "mb_match_encode": (C.c_int, [_p, _i64, _p, _i64, _f32, _f32, _i32, _f32, _f32, _f32, _f32, _p, _p, _p, _p, _sz, _p]),
    "mb_roi_align_backward": (C.c_int, [_p, _p, _i64, _f32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p]),
    "mb_paste_masks": (C.c_int, [_p, _p, _i64, _i32, _i32, _i32, _i32, _p, _p]),
    "mb_mask_prob": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _p]),
    "mb_crop_masks": (C.c_int, [C.POINTER(CropParams), _p, _p, _i32, _i32, _p, _i32, _f32, _p, _p, _p, _p, _p, _i64, _p]),
    "mb_image_transform": (C.c_int, [C.POINTER(TransformParams), _p, _p]),
}

_lib = None
_lock = threading.Lock()


class MisoB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libmisob200.so and bind every symbol of the ABI. Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise MisoB200Error(
                f"{LIB_PATH} not found: build it with `python -m miso_b200.build` "
                "(nvcc, sm_100a). miso_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if lib.mb_abi_version() != 1:
            raise MisoB200Error("libmisob200.so ABI version mismatch; rebuild")
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc == MB_OK:
        return
    if rc < 0:
        raise MisoB200Error(f"{what}: {MB_ERRORS.get(rc, rc)}")
    raise MisoB200Error(f"{what}: CUDA error {rc}")
