"""ctypes binding of ``libssd3d_b200.so`` (C ABI declared in ``include/ssd3d_b200.h``).

There is deliberately no fallback: if the CUDA library is missing or an entry point is absent the
import of the ops fails loudly, so a "passing" run can never be a silent PyTorch/CPU path.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libssd3d_b200.so")

SSD3D_OK = 0
SSD3D_ERR_ARG = 10001
SSD3D_ERR_TMA = 10002
SSD3D_ERR_UNSUPPORTED = 10003
NAN_BACKBONE, NAN_LOCS, NAN_SCORES = 1, 2, 4
SORT_MAX = 16384
NMS_NO_GRID = 1
BOX_CXCYCZ_TO_XYZ, BOX_XYZ_TO_CXCYCZ, BOX_GCXGCYGCZ_TO_CXCYCZ, BOX_CXCYCZ_TO_GCXGCYGCZ = 0, 1, 2, 3

P = c_void_p  # every device pointer / stream crosses the ABI as a plain address

MAX_PRIOR_LAYERS, MAX_PRIOR_SIZES = 8, 4


class PriorTable(ctypes.Structure):
    """``ssd3d_prior_table`` of include/ssd3d_b200.h (prior boxes as a closed-form function of the prior index)."""
    _fields_ = [("n_layers", c_int32),
                ("d0", c_int32 * MAX_PRIOR_LAYERS), ("d1", c_int32 * MAX_PRIOR_LAYERS), ("d2", c_int32 * MAX_PRIOR_LAYERS),
                ("n_boxes", c_int32 * MAX_PRIOR_LAYERS), ("pad_", c_int32),
                ("start", c_int64 * (MAX_PRIOR_LAYERS + 1)),
                ("size", (c_float * MAX_PRIOR_SIZES) * MAX_PRIOR_LAYERS)]

# name -> (restype, argtypes); mirrors include/ssd3d_b200.h one to one
SIGNATURES = {
    "ssd3d_version": (c_char_p, []),
    "ssd3d_stem_conv_bn_relu": (c_int, [P, c_int, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_stem_conv_bn_relu_simt": (c_int, [P, c_int, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_stem_tc_supported": (c_int, [c_int, c_int, c_int]),
    "ssd3d_dwconv3d_bn_relu": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_block_fused_supported": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "ssd3d_block_dwpw_bn_relu": (c_int, [P, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P]),
    "ssd3d_pwconv_bn_relu": (c_int, [P, P, P, P, P, c_int64, c_int, c_int, P, P]),
    "ssd3d_head_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "ssd3d_head_conv": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int64,
                                c_int64, P, P, c_int64, c_int, P]),
    "ssd3d_head_weight_kw": (c_int, [P, c_int, P, P]),
    "ssd3d_head_kw_supported": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "ssd3d_box_transform": (c_int, [c_int, P, P, P, c_int64, P]),
    "ssd3d_iou3d_pairwise": (c_int, [P, P, P, c_int64, c_int64, c_int, P]),
    "ssd3d_detect_workspace_bytes": (c_int64, [c_int, c_int64, c_int, c_int]),
    "ssd3d_detect_objects": (c_int, [P, P, P, c_int, c_int64, c_int, c_float, c_float, c_int, P, P, P, P, P, P,
                                     c_int64, P, P]),
    "ssd3d_decode_softmax": (c_int, [P, P, P, c_int, c_int64, c_int, P, P, P]),
    "ssd3d_nms3d_sorted": (c_int, [P, c_int64, c_float, P, P, P]),
    "ssd3d_nms3d_chunked_workspace_bytes": (c_int64, [c_int64, c_int]),
    "ssd3d_nms3d_sorted_chunked": (c_int, [P, c_int64, c_float, P, P, P, c_int64, c_int, c_int, P]),
    "ssd3d_sort_keys_u64": (c_int, [P, c_int64, P, P]),
    "ssd3d_decode_filter": (c_int, [P, P, P, c_int, c_int64, c_int, c_float, P, P, P, P]),
    "ssd3d_match_priors": (c_int, [P, P, P, c_int, c_int64, P, c_int64, c_float, c_float, P, P, P, P, P, P, P]),
    "ssd3d_multibox_workspace_bytes": (c_int64, [c_int, c_int64]),
    "ssd3d_multibox_loss": (c_int, [P, P, P, P, c_int, c_int64, c_int, c_float, c_int, c_int, P, P, P, P, P,
                                    c_int64, P]),
    # ---- training step ----
    "ssd3d_stem_conv_affine": (c_int, [P, c_int, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_stem_conv_affine_simt": (c_int, [P, c_int, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_stem_conv_affine_tz": (c_int, [P, c_int, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_stem_tz_supported": (c_int, [c_int, c_int, c_int]),
    "ssd3d_stem_dw_fused": (c_int, [P, c_int, P, P, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_stem_dw_fused_supported": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int]),
    "ssd3d_stem_conv_affine_tc": (c_int, [P, c_int, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_dwconv3d_affine": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_dwconv3d_affine_direct": (c_int, [P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_pwconv_affine": (c_int, [P, P, P, P, P, c_int64, c_int, c_int, c_int, P, P]),
    "ssd3d_bn_workspace_bytes": (c_int64, [c_int]),
    "ssd3d_bn_train_fwd": (c_int, [P, c_int64, c_int, P, P, c_float, c_float, P, P, P, P, P, P, P, P, P, P, c_int64, P]),
    "ssd3d_gather_cast": (c_int, [P, P, c_int64, P, c_int, P]),
    "ssd3d_normalize_workspace_bytes": (c_int64, [c_int]),
    "ssd3d_normalize_intensity_nonzero": (c_int, [P, c_int, c_int64, P, c_int, P, c_int64, P]),
    "ssd3d_gt_boxes_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "ssd3d_gt_boxes_from_segmentation": (c_int, [P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P,
                                                 c_int64, P]),
    "ssd3d_gt_boxes_instances_workspace_bytes": (c_int64, [c_int, c_int, c_int]),
    "ssd3d_gt_boxes_from_instances": (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, c_int, c_int, c_int, P, P, P,
                                              P, P, c_int64, P]),
    "ssd3d_bn_relu_bwd": (c_int, [P, P, c_int64, c_int, P, P, P, P, P, P, P, P, c_int64, P]),
    "ssd3d_bn_unit_supported": (c_int, [c_int64, c_int]),
    "ssd3d_bn_unit_workspace_bytes": (c_int64, [c_int]),
    "ssd3d_bn_unit_fwd": (c_int, [P, c_int64, c_int, P, P, c_float, c_float, P, P, P, P, P, P, P, P, P, P, c_int64, P,
                                  P]),
    "ssd3d_bn_unit_bwd": (c_int, [P, P, c_int64, c_int, P, P, P, P, P, P, P, P, c_int64, P, P]),
    "ssd3d_wgrad_workspace_bytes": (c_int64, [c_int64, c_int, c_int]),
    "ssd3d_pwconv_wgrad": (c_int, [P, P, c_int64, c_int, c_int, P, P, c_int64, P]),
    "ssd3d_stem_wgrad": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, c_int64, P]),
    "ssd3d_stem_wgrad_bn": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, P, P, P, P, P,
                                    c_int64, P]),
    "ssd3d_head_wgrad": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, P, P, P, c_int64, P]),
    "ssd3d_head_grad_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int, c_int]),
    "ssd3d_head_grad_pack": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, c_int64, P, P, P, P,
                                     c_int64, P]),
    "ssd3d_head_dgrad": (c_int, [P, P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_dwconv3d_dgrad": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, c_int, P]),
    "ssd3d_dw_wgrad_workspace_bytes": (c_int64, [c_int]),
    "ssd3d_dwconv3d_wgrad": (c_int, [P, P, c_int, c_int, c_int, c_int, c_int, c_int, P, P, c_int64, P]),
    "ssd3d_map_workspace_bytes": (c_int64, [c_int64, c_int64]),
    "ssd3d_map_class": (c_int, [P, P, P, c_int64, P, P, P, c_int64, c_float, P, c_int, P, P, P, P, P, P, P, P, P, P,
                                c_int64, P]),
    "ssd3d_adam_step": (c_int, [P, P, P, P, c_int64, c_int64, c_float, c_float, c_float, c_float, c_float, c_float,
                                c_int, c_float, P, P]),
    "ssd3d_generate_volumes": (c_int, [ctypes.c_uint64, c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_int, c_int, P, P, P, P, P]),
    "ssd3d_prior_boxes": (c_int, [P, c_int64, P, P]),
    "ssd3d_decode_softmax_analytic": (c_int, [P, P, P, c_int, c_int64, c_int, P, P, P]),
    "ssd3d_decode_filter_analytic": (c_int, [P, P, P, c_int, c_int64, c_int, c_float, P, P, P, P]),
    "ssd3d_detect_objects_analytic": (c_int, [P, P, P, c_int, c_int64, c_int, c_float, c_float, c_int, P, P, P, P, P,
                                              P, c_int64, P, P]),
    "ssd3d_match_priors_analytic": (c_int, [P, P, P, c_int, c_int64, P, c_int64, c_float, c_float, P, P, P, P, P, P,
                                            P]),
    "ssd3d_adam_step_dev": (c_int, [P, P, P, P, c_int64, c_int64, c_float, c_float, c_int, c_float, c_float, c_float,
                                    c_float, c_float, P, P, P]),
    # ---- training batches from a device-resident data set ----
    "ssd3d_augment_batch": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P, c_int, c_int, c_int,
                                    c_int, c_float, c_float, c_float, c_int, c_int, c_float, c_float, P, P, P, P]),
    "ssd3d_gt_pack": (c_int, [P, P, P, P, c_int, c_int, c_int, P, P, P, P, P]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the library once and attach the prototypes; raise if it (or any symbol) is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "%s not found: build it with `python -m mslesions3d_b200.build` (needs nvcc; no CPU fallback exists)"
            % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code: int, what: str) -> None:
    if code == SSD3D_OK:
        return
    names = {SSD3D_ERR_ARG: "invalid argument", SSD3D_ERR_TMA: "TMA descriptor creation failed",
             SSD3D_ERR_UNSUPPORTED: "unsupported configuration"}
    if code in names:
        raise RuntimeError("%s: %s (code %d)" % (what, names[code], code))
    raise RuntimeError("%s: CUDA error %d" % (what, code))
