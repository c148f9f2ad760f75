"""ctypes binding of the C-ABI in include/hd_yolo_b200.h.

The shared library is built in-tree by ``hd_yolo_b200/csrc/build.sh`` (or
``__graft_entry__.build()``).  There is no CPU fallback and no alternative
backend: if the library is missing, or a call fails, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HDY_MAX_LEVELS = 8
HDY_MAX_ANCHORS = 8
HDY_MAX_SCORES = 96
HDY_STATUS_OVERFLOW = 1
HDY_STATUS_ROUNDS = 2
HDY_F32, HDY_F16 = 0, 1
HDY_SEAM_HDR_WORDS, HDY_SEAM_FAR_WORDS, HDY_SEAM_ROW_WORDS, HDY_SEAM_META_WORDS, HDY_SEAM_MAX_WORLD = 16, 8, 6, 96, 64

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhdyolo_b200.so")


class HdyError(RuntimeError):
    pass


class Level(C.Structure):
    """hdy_level_t"""

    _fields_ = [
        ("logits", C.c_void_p),
        ("ny", C.c_int32),
        ("nx", C.c_int32),
        ("stride", C.c_float),
        ("anchor_w", C.c_float * HDY_MAX_ANCHORS),
        ("anchor_h", C.c_float * HDY_MAX_ANCHORS),
        ("dtype", C.c_int32),
    ]


class FeatureLevel(C.Structure):
    """hdy_feature_level_t"""

    _fields_ = [("data", C.c_void_p), ("h", C.c_int32), ("w", C.c_int32), ("spatial_scale", C.c_float)]


_vp, _i, _f, _sz, _i64 = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64
_LP = C.POINTER(Level)

# name -> (restype, argtypes); must list every symbol the header declares
SIGNATURES = {
    "hdy_version": (C.c_char_p, []),
    "hdy_last_error": (C.c_char_p, []),
    "hdy_device_sm_count": (_i, []),
    "hdy_zero_i32": (_i, [_vp, _sz, _vp]),
    "hdy_decode_levels": (_i, [_LP, _i, _i, _i, _i, C.POINTER(_vp), _vp]),
    "hdy_decode_concat": (_i, [_LP, _i, _i, _i, _i, _i, _vp, _vp]),
    "hdy_filter_compact_logits": (_i, [_LP, _i, _i, _i, _i, _i, _i, _f, _f, _i, _vp, _vp, _vp, _vp, _vp]),
    "hdy_filter_compact_preds": (_i, [_vp, _i, _i, _i, _f, _f, _i, _vp, _vp, _vp, _vp, _vp]),
    "hdy_filter_compact_yolo": (_i, [_vp, _i, _i, _i, _f, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hdy_nms_workspace_bytes": (_sz, [_i, _i]),
    "hdy_nms_tiles": (
        _i,
        [_vp, _vp, _vp, _vp, _i, _i, _f, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _sz, _vp],
    ),
    "hdy_make_keys": (_i, [_vp, _i, _i, _vp, _vp]),
    "hdy_debug_nms_phases": (_i, [_vp]),
    "hdy_gather_preds": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp]),
    "hdy_gather_logits": (_i, [_LP, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "hdy_gather_select_logits": (_i, [_LP, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, C.POINTER(C.c_int32), _i, _f, _vp, _vp,
                                      _vp, _vp, _vp, _vp]),
    "hdy_select_scores": (_i, [_vp, _vp, _i, _i, _i, C.POINTER(C.c_int32), _i, _f, _vp, _vp, _vp]),
    "hdy_mask_select": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "hdy_paste_masks": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "hdy_paste_geometry": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "hdy_paste_masks_packed": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, C.c_int64, _vp, _vp]),
    "hdy_unpack_masks": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "hdy_process_mask_workspace_bytes": (_sz, [_i, _i]),
    "hdy_process_mask": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "hdy_process_mask_geometry": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "hdy_process_mask_rows": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "hdy_process_mask_packed": (
        _i,
        [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, C.c_int64, _vp, _vp, _sz, _vp],
    ),
    "hdy_affine_boxes": (_i, [_vp, _i64, _i, _f, _f, _f, _f, _f, _f, _i, _vp]),
    "hdy_merge_append": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                              _vp]),
    "hdy_merge_overhang": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "hdy_merge_overhang_cap": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _f, _f, _vp, _vp, _vp]),
    "hdy_merge_dirty_tiles": (_i, [_vp, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "hdy_merge_workspace_bytes": (_sz, [_i64]),
    "hdy_merge_nms": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "hdy_merge_rounds": (_i, [_vp, _i64, _f, _i, _i, _vp]),
    "hdy_merge_finish": (_i, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "hdy_seam_summary": (_i, [_vp, _i64, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "hdy_seam_select": (_i, [_vp, _vp, _i64, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "hdy_seam_scatter": (_i, [_vp, _vp, _i, _i, _i, _i, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hdy_seam_dirty_tiles": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp]),
    "hdy_seam_build": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i64, _i64, _f, _f, _vp, _vp, _sz, _vp]),
    "hdy_seam_export": (_i, [_vp, _i64, _vp, _vp, _vp, _i, _vp, _vp]),
    "hdy_seam_import": (_i, [_vp, _i64, _i64, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "hdy_sort_workspace_bytes": (_sz, [_i64]),
    "hdy_sort_keys_bytes": (_i, [_vp, _vp, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "hdy_merge_select_ordered": (_i, [_vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "hdy_rcnn_decode": (_i, [_vp, _vp, _i64, _i, _i64, _f, _f, _f, _f, _f, _vp, _vp]),
    "hdy_softmax_rows": (_i, [_vp, _i64, _i, _vp, _vp]),
    "hdy_rcnn_filter_compact": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i, _f, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hdy_rpn_level_keys": (_i, [_vp, _i, _i, C.POINTER(C.c_int32), _i, _vp, _vp]),
    "hdy_rpn_topk_compact": (_i, [_vp, _vp, _i, _i, C.POINTER(C.c_int32), _i, _i, _vp, _f, _f, _i, _i, _vp, _vp, _vp,
                                  _vp, _vp, _vp]),
    "hdy_regroup_kept": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hdy_merge_gather": (_i, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hdy_multiscale_roi_align": (_i, [C.POINTER(FeatureLevel), _i, _i, _i, _vp, _vp, _i64, _i, _i, _i, _vp, _vp]),
    "hdy_multiscale_roi_align_tf32x3": (_i, [C.POINTER(FeatureLevel), _i, _i, _i, _i, _vp, _vp, _i64, _i, _i, _i, _vp,
                                            _vp, _vp]),
    "hdy_match_pairs": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp, _i, _f, _i, _vp, _vp, _vp, _vp, _vp]),
    "hdy_box_iou": (_i, [_vp, _i64, _vp, _i64, _vp, _vp]),
}

_lock = threading.Lock()
_lib = None


def load():
    """Load (once) and return the ctypes handle; raises HdyError if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise HdyError(
                f"{LIB_PATH} is missing: build it with `bash hd_yolo_b200/csrc/build.sh` "
                "(or `python -c 'import __graft_entry__ as g; g.build()'`). "
                "hd_yolo_b200 has no CPU or PyTorch fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:  # pragma: no cover
                raise HdyError(f"{LIB_PATH} does not export {name}; rebuild it") from e
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().hdy_last_error().decode("utf-8", "replace")
        raise HdyError(f"{what or 'hdy call'} failed (rc={rc}): {msg}")


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
