"""ctypes binding of libdgod_b200.so — the C ABI declared in include/dgod_b200.h.

There is no CPU fallback: if the library is missing and cannot be built, importing any op fails
loudly.  The `.so` is built in-tree (dgod_b200/build.py) so it ships with the repo snapshot.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libdgod_b200.so"

MAX_LEVELS = 8
MAX_CELL_ANCHORS = 16
F32, BF16 = 0, 1
ABI_VERSION = 9   # DGOD_ABI_VERSION of include/dgod_b200.h

vp, i32, i64, f32, f64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t


class RpnConfig(C.Structure):
    """dgod_rpn_config (include/dgod_b200.h)."""
    _fields_ = [
        ("n_img", i32), ("n_levels", i32), ("anchors_per_loc", i32),
        ("height", i32 * MAX_LEVELS), ("width", i32 * MAX_LEVELS),
        ("stride_h", i32 * MAX_LEVELS), ("stride_w", i32 * MAX_LEVELS),
        ("cell_anchors", ((f32 * 4) * MAX_CELL_ANCHORS) * MAX_LEVELS),
        ("pre_nms_top_n", i32), ("post_nms_top_n", i32),
        ("nms_thresh", f64),
        ("min_size", f32), ("score_thresh", f32), ("bbox_xform_clip", f32),
    ]


class RoiConfig(C.Structure):
    """dgod_roi_config (include/dgod_b200.h)."""
    _fields_ = [
        ("n_levels", i32), ("batch", i32), ("channels", i32),
        ("height", i32 * MAX_LEVELS), ("width", i32 * MAX_LEVELS),
        ("spatial_scale", f32 * MAX_LEVELS),
        ("channels_last", i32), ("dtype", i32),
        ("pooled_h", i32), ("pooled_w", i32), ("sampling_ratio", i32), ("aligned", i32),
        ("k_min", i32), ("k_max", i32),
        ("canonical_scale", f32), ("canonical_level", f32), ("eps", f32),
    ]


# name -> (restype, argtypes); must list every function declared in include/dgod_b200.h
SIGNATURES = {
    "dgod_abi_version": (i32, []),
    "dgod_last_error": (C.c_char_p, []),
    "dgod_launch_count": (C.c_uint64, []),
    "dgod_box_iou": (i32, [vp, i32, vp, i32, vp, vp]),
    "dgod_matcher_workspace_bytes": (sz, [i32]),
    "dgod_matcher": (i32, [vp, i32, i32, f64, f64, i32, vp, vp, sz, vp]),
    "dgod_iou_match_workspace_bytes": (sz, [i32, i32]),
    "dgod_iou_match": (i32, [vp, vp, vp, i32, i32, vp, vp, vp, i32, i32, f64, f64, i32,
                             vp, vp, vp, vp, vp, vp, sz, vp]),
    "dgod_fcos_assign": (i32, [vp, i32, i32, i32, f64, vp, vp, vp, i32, vp, vp, vp, vp, i32, vp]),
    "dgod_fcos_loss_workspace_bytes": (sz, [C.c_longlong]),
    "dgod_fcos_loss_fwd": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, vp, vp, sz, vp]),
    "dgod_fcos_loss_bwd": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, vp, vp, vp, vp, vp, vp]),
    "dgod_fcos_candidates": (i32, [vp, vp, vp, vp, i32, i32, vp, i32, i32, vp, f32, i32, vp, vp, vp, vp, vp, vp]),
    "dgod_balanced_sample": (i32, [vp, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]),
    "dgod_sample_rois": (i32, [vp, vp, i32, vp, vp, i32, vp, vp, i32, i32, vp, vp, i32, vp, vp, i32, f32, f32, f32, f32,
                               vp, vp, vp, vp]),
    "dgod_nms_workspace_bytes": (sz, [i32, i32, i32]),
    "dgod_nms_batched": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, f64, i32, i32, vp, vp, vp, vp, sz, vp]),
    "dgod_rpn_workspace_bytes": (sz, [C.POINTER(RpnConfig)]),
    "dgod_rpn_proposals": (i32, [C.POINTER(RpnConfig), C.POINTER(vp), C.POINTER(vp), vp, vp, vp, vp, vp, sz, vp]),
    "dgod_rpn_filter": (i32, [C.POINTER(RpnConfig), vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "dgod_msroi_align_fwd_workspace_bytes": (sz, [i32]),
    "dgod_msroi_align_fwd": (i32, [C.POINTER(RoiConfig), C.POINTER(vp), vp, i32, vp, vp, sz, vp]),
    "dgod_msroi_align_bwd_workspace_bytes": (sz, [i32]),
    "dgod_msroi_align_bwd_workspace_bytes_cfg": (sz, [C.POINTER(RoiConfig), i32]),
    "dgod_msroi_align_bwd": (i32, [C.POINTER(RoiConfig), vp, vp, i32, vp, C.POINTER(vp), i32, vp, sz, vp]),
    "dgod_box_decode": (i32, [vp, vp, i32, i32, f32, f32, f32, f32, f32, vp, vp]),
    "dgod_detect_candidates": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, f32, f32, f32, f32, f32,
                                     f32, f32, vp, vp, vp, vp, vp]),
    "dgod_grl_scale": (i32, [vp, vp, i64, f32, i32, vp]),
    "dgod_image_batch": (i32, [C.POINTER(vp), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), i32, i32,
                               C.POINTER(f32), C.POINTER(f32), vp, i32, i32, vp]),
    "dgod_image_batch_u8": (i32, [C.POINTER(vp), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), i32, i32,
                                  C.POINTER(f32), C.POINTER(f32), vp, i32, i32, vp]),
    "dgod_nchw_to_nhwc": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "dgod_fpn_merge_fwd": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dgod_fpn_merge_bwd": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dgod_stem_pool_fwd": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dgod_shift_relu_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dgod_bias_add_fwd": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dgod_fpn_merge_fwd_bf16": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dgod_fpn_merge_bwd_bf16": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dgod_stem_pool_fwd_bf16": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "dgod_shift_relu_fwd_bf16": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "dgod_map_match": (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, i32, i32, vp, vp, vp]),
    "dgod_map_accumulate_workspace_bytes": (sz, [i32, i32]),
    "dgod_map_accumulate": (i32, [vp, vp, vp, i32, i32, vp, i32, i32, vp, vp, vp, sz, vp]),
    "dgod_linear_tc_workspace_bytes": (sz, [i32, i32, i32]),
    "dgod_linear_tc": (i32, [vp, i32, vp, i32, i32, i32, i32, vp, i32, vp, vp, vp, sz, vp]),
    "dgod_rpn_head_workspace_bytes": (sz, []),
    "dgod_rpn_head_fwd": (i32, [C.POINTER(vp), i32, C.POINTER(i32), C.POINTER(i32), i32, i32, i32, vp, vp, vp, vp, vp,
                                C.POINTER(vp), C.POINTER(vp), vp]),
    "dgod_rpn_head_bwd": (i32, [C.POINTER(vp), i32, C.POINTER(i32), C.POINTER(i32), i32, i32, i32, vp, vp, vp,
                                C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), vp, vp, sz, vp]),
}

_lib = None


class DgodError(RuntimeError):
    pass


def load():
    """Returns the loaded library; builds it with nvcc first if it is missing (dev boxes)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists() or os.environ.get("DGOD_REBUILD"):
        try:
            from .build import build
            build()
        except Exception as e:  # pragma: no cover - depends on the toolchain
            raise DgodError(
                f"dgod_b200: {LIB_PATH} is missing and could not be built ({e}). "
                "There is no CPU fallback: run `python -c 'import __graft_entry__ as g; g.build()'`."
            ) from e
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.dgod_abi_version() != ABI_VERSION:
        raise DgodError("dgod_b200: ABI version mismatch between _lib.py and libdgod_b200.so")
    _lib = lib
    return lib


def check(rc: int, exc=RuntimeError):
    if rc != 0:
        msg = load().dgod_last_error().decode("utf-8", "replace")
        raise exc(msg if msg else f"dgod_b200 call failed with code {rc}")


def launch_count() -> int:
    return int(load().dgod_launch_count())
