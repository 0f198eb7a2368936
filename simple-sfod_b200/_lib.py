"""ctypes binding of libsfod_b200.so (the C ABI declared in include/sfod_b200.h).

There is NO fallback for the operators of this library: if the shared library is missing or a call fails, an exception is
raised, and every operator of ``ops`` refuses CPU tensors.  (The one place where another implementation runs is an operator
boundary, not a fallback: ``modeling.SfodBatchNorm2d`` hands the modes the kernels do not serve -- autograd, eval, CPU -- to
PyTorch's own ``nn.BatchNorm2d``, as documented there.)  The product path never imports anything from ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsfod_b200.so")
_lib: Optional[C.CDLL] = None

c_f32p = C.c_void_p  # device pointers are passed as raw addresses
c_ptr = C.c_void_p


class EmaTensor(C.Structure):
    _fields_ = [("student", C.c_void_p), ("teacher", C.c_void_p), ("numel", C.c_int64), ("dtype", C.c_int32),
                ("reserved", C.c_int32)]


class JitterParams(C.Structure):
    _fields_ = [("n_ops", C.c_int32), ("op", C.c_int32 * 4), ("factor", C.c_float * 4), ("hue_shift", C.c_int32 * 4), ("grayscale", C.c_int32)]


class EraseParams(C.Structure):
    _fields_ = [("n_rects", C.c_int32), ("rect", (C.c_int32 * 4) * 4)]


class ResizeImage(C.Structure):
    _fields_ = [("src", C.c_void_p), ("stride_row", C.c_int64), ("stride_px", C.c_int64), ("stride_ch", C.c_int64),
                ("in_h", C.c_int32), ("in_w", C.c_int32), ("out_h", C.c_int32), ("out_w", C.c_int32), ("out_offset", C.c_int64),
                ("hflip", C.c_int32), ("kx_offset", C.c_int32), ("kx_size", C.c_int32), ("ky_offset", C.c_int32),
                ("ky_size", C.c_int32), ("reserved", C.c_int32)]


class RpnParams(C.Structure):
    _fields_ = [("N", C.c_int), ("HWA", C.c_int), ("A", C.c_int), ("Hf", C.c_int), ("Wf", C.c_int), ("stride", C.c_int),
                ("anchor_offset", C.c_float), ("weights", C.c_float * 4), ("scale_clamp", C.c_float),
                ("pre_nms_topk", C.c_int), ("post_nms_topk", C.c_int), ("min_box_size", C.c_float),
                ("nms_thresh", C.c_double), ("cell_anchors", C.c_float * 256), ("head_layout", C.c_int)]


class FrcnnParams(C.Structure):
    _fields_ = [("N", C.c_int), ("R", C.c_int), ("K", C.c_int), ("class_agnostic", C.c_int),
                ("max_rows_per_image", C.c_int), ("weights", C.c_float * 4), ("scale_clamp", C.c_float),
                ("score_thresh", C.c_float), ("nms_thresh", C.c_double), ("topk", C.c_int), ("pseudo_thresh", C.c_float),
                ("coord_trick_max_n", C.c_int64), ("rows_stride", C.c_int)]


COCO_MAX_CATEGORIES, COCO_MAX_IOU_THRS, COCO_MAX_REC_THRS, COCO_MAX_AREA_RNGS, COCO_MAX_MAX_DETS = 254, 16, 128, 4, 4


class CocoEvalParams(C.Structure):
    _fields_ = [("n_images", C.c_int32), ("n_categories", C.c_int32), ("dt_stride", C.c_int32), ("n_iou_thrs", C.c_int32),
                ("n_rec_thrs", C.c_int32), ("n_area_rngs", C.c_int32), ("n_max_dets", C.c_int32),
                ("max_dets", C.c_int32 * COCO_MAX_MAX_DETS), ("reserved", C.c_int32), ("iou_thrs", C.c_double * COCO_MAX_IOU_THRS),
                ("rec_thrs", C.c_double * COCO_MAX_REC_THRS), ("area_rng", (C.c_double * 2) * COCO_MAX_AREA_RNGS)]


P2P_MAX_RANKS = 8
P2P_HANDLE_BYTES = 64


class P2PComm(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("inbox", C.c_void_p * P2P_MAX_RANKS)]


# sfod_abi_version() of the library this binding is written for, and the struct mirrors in the order of sfod_abi_sizeof(which)
ABI_VERSION = 3
ABI_STRUCTS = (EmaTensor, RpnParams, FrcnnParams, P2PComm, JitterParams, EraseParams, ResizeImage, CocoEvalParams)


# name -> (restype, argtypes); every symbol include/sfod_b200.h declares
SIGNATURES = {
    "sfod_abi_version": (C.c_int, []),
    "sfod_abi_sizeof": (C.c_size_t, [C.c_int]),
    "sfod_status_string": (C.c_char_p, [C.c_int]),
    "sfod_debug_launch_count": (C.c_uint64, []),
    "sfod_ema_plan_chunks": (C.c_int64, [C.POINTER(EmaTensor), C.c_int]),
    "sfod_ema_plan_bytes": (C.c_size_t, [C.c_int64]),
    "sfod_ema_plan_build": (C.c_int, [C.POINTER(EmaTensor), C.c_int, c_ptr, C.c_size_t]),
    "sfod_ema_multi_tensor": (C.c_int, [c_ptr, C.c_int64, C.c_double, c_ptr]),
    "sfod_roi_align_fwd_workspace_bytes": (C.c_size_t, [C.c_int] * 7),
    "sfod_roi_align_fwd": (C.c_int, [c_ptr, C.c_int, c_ptr] + [C.c_int] * 7 + [C.c_float, C.c_int, C.c_int, C.c_int, c_ptr,
                                     c_ptr, C.c_size_t, c_ptr]),
    "sfod_roi_align_bwd_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "sfod_roi_align_bwd": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 7 + [C.c_float, C.c_int, C.c_int, c_ptr, C.c_int, c_ptr,
                                     C.c_size_t, c_ptr]),
    "sfod_roi_pool_fwd": (C.c_int, [c_ptr, c_ptr] + [C.c_int] * 7 + [C.c_float, c_ptr, c_ptr, c_ptr]),
    "sfod_roi_pool_bwd": (C.c_int, [c_ptr, c_ptr, c_ptr] + [C.c_int] * 7 + [c_ptr, c_ptr]),
    "sfod_nms_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "sfod_nms": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int64, C.c_double, C.c_int64, c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "sfod_rpn_select_workspace_bytes": (C.c_size_t, [C.POINTER(RpnParams)]),
    "sfod_rpn_select": (C.c_int, [C.POINTER(RpnParams)] + [c_ptr] * 10 + [C.c_size_t, c_ptr]),
    "sfod_frcnn_postprocess_workspace_bytes": (C.c_size_t, [C.POINTER(FrcnnParams)]),
    "sfod_frcnn_postprocess": (C.c_int, [C.POINTER(FrcnnParams)] + [c_ptr] * 14 + [C.c_size_t, c_ptr]),
    "sfod_apply_deltas": (C.c_int, [c_ptr, c_ptr, C.c_int64, C.c_int, C.POINTER(C.c_float), C.c_float, c_ptr, c_ptr]),
    "sfod_softmax_lastdim": (C.c_int, [c_ptr, C.c_int64, C.c_int, c_ptr, c_ptr]),
    "sfod_threshold_select": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_float, c_ptr, c_ptr, c_ptr]),
    "sfod_class_threshold_select": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr]),
    "sfod_class_histogram": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_float, c_ptr, c_ptr]),
    "sfod_normalize_pad": (C.c_int, [c_ptr, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                     C.c_int, C.c_int, C.c_int, c_ptr, c_ptr]),
    "sfod_iou_match_workspace_bytes": (C.c_size_t, [C.c_int]),
    "sfod_iou_match": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_int), C.c_int, C.c_int,
                                 c_ptr, c_ptr, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "sfod_color_jitter_pil": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, C.c_size_t, c_ptr, c_ptr]),
    "sfod_gaussian_blur_pil": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, C.c_int, c_ptr, c_ptr]),
    "sfod_random_erase": (C.c_int, [c_ptr, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, C.c_uint64, c_ptr]),
    "sfod_resize_pil": (C.c_int, [c_ptr, C.c_int, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, c_ptr]),
    "sfod_linear_3xtf32_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.c_int]),
    "sfod_linear_3xtf32": (C.c_int, [c_ptr, C.c_int64, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int, c_ptr, c_ptr, C.c_size_t, c_ptr]),
    "sfod_coco_eval_workspace_bytes": (C.c_size_t, [C.POINTER(CocoEvalParams)]),
    "sfod_coco_eval": (C.c_int, [C.POINTER(CocoEvalParams)] + [c_ptr] * 14 + [C.c_size_t, c_ptr]),
    "sfod_subsample_labels": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_uint64, c_ptr, c_ptr, c_ptr]),
    "sfod_bn_stats_bytes": (C.c_size_t, [C.c_int]),
    "sfod_bn_partial_stats": (C.c_int, [c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int64, c_ptr, C.POINTER(P2PComm), c_ptr]),
    "sfod_bn_finalize_apply": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, C.POINTER(P2PComm),
                                         c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, C.c_double, C.c_double, C.c_int, C.c_int, c_ptr]),
    "sfod_bn_train_fused": (C.c_int, [c_ptr, c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr,
                                      C.c_double, C.c_double, C.c_int, c_ptr]),
    "sfod_bn_frozen_scratch_bytes": (C.c_size_t, [C.c_int]),
    "sfod_bn_frozen_apply": (C.c_int, [c_ptr, c_ptr, c_ptr, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, c_ptr, c_ptr,
                                       C.c_double, C.c_int, c_ptr, c_ptr]),
    "sfod_p2p_inbox_bytes": (C.c_size_t, []),
    "sfod_p2p_max_channels": (C.c_int, []),
    "sfod_p2p_alloc": (C.c_int, [C.POINTER(C.c_void_p), c_ptr]),
    "sfod_p2p_open": (C.c_int, [c_ptr, C.POINTER(C.c_void_p)]),
    "sfod_p2p_close": (C.c_int, [c_ptr]),
    "sfod_p2p_free": (C.c_int, [c_ptr]),
    "sfod_p2p_status": (C.c_int, [C.POINTER(P2PComm), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
}


class SfodLibraryError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load libsfod_b200.so (built by simple-sfod_b200/build.py).  Raises if it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SfodLibraryError(
                f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first. "
                "There is no CPU fallback for the sfod_b200 hot path.")
        try:
            import torch  # noqa: F401  (loads the CUDA runtime the library links against)
        except Exception:  # pragma: no cover
            pass
        try:
            handle = C.CDLL(LIB_PATH)
        except OSError as e:
            raise SfodLibraryError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _check_abi(handle)
        _lib = handle
    return _lib


def _check_abi(handle: C.CDLL) -> None:
    """Refuse a library built from another revision of the header: ctypes would hand it argument lists it does not expect."""
    version = handle.sfod_abi_version()
    if version != ABI_VERSION:
        raise SfodLibraryError(f"{LIB_PATH} has ABI version {version}, this binding expects {ABI_VERSION}: rebuild it "
                               "(`python simple-sfod_b200/build.py --force`)")
    for which, mirror in enumerate(ABI_STRUCTS):
        size = handle.sfod_abi_sizeof(which)
        if size != C.sizeof(mirror):
            raise SfodLibraryError(f"{LIB_PATH}: struct {which} has {size} bytes, its ctypes mirror {mirror.__name__} {C.sizeof(mirror)}")


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = lib().sfod_status_string(int(status)).decode()
        raise SfodLibraryError(f"libsfod_b200 {what} failed with status {status}: {msg}")
