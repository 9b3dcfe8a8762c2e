"""ctypes binding of include/yolonano_b200.h.

There is deliberately no fallback: if the shared library is missing or a symbol the
header declares cannot be resolved, importing the product path raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libyolonano_b200.so"

YNB_ABI_VERSION = 1
YNB_OK = 0
GEMM_FP32_FFMA, GEMM_TC_3XTF32, GEMM_TC_TF32, GEMM_TC_BF16 = 0, 1, 2, 3


class YnbConfig(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("device", C.c_int32),
        ("input_size", C.c_int32),
        ("num_classes", C.c_int32),
        ("num_anchors", C.c_int32),
        ("anchors", C.c_float * 18),
        ("conf_thresh", C.c_float),
        ("nms_thresh", C.c_float),
        ("diou_nms", C.c_int32),
        ("gemm_mode", C.c_int32),
        ("max_batch", C.c_int32),
    ]


_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f = C.c_float
_s = C.c_char_p

# name -> (restype, argtypes): every symbol of include/yolonano_b200.h
SIGNATURES = {
    "ynb_create": (C.c_int, [C.POINTER(YnbConfig), C.POINTER(_p)]),
    "ynb_destroy": (None, [_p]),
    "ynb_last_error": (_s, [_p]),
    "ynb_abi_version": (C.c_int, []),
    "ynb_set_grid": (C.c_int, [_p, _i32]),
    "ynb_set_thresholds": (C.c_int, [_p, _f, _f, _i32]),
    "ynb_set_gemm_mode": (C.c_int, [_p, _i32]),
    "ynb_num_boxes": (_i64, [_p]),
    "ynb_workspace_bytes": (_i64, [_p, _i32]),
    "ynb_num_convs": (_i32, []),
    "ynb_conv_name": (_s, [_i32]),
    "ynb_conv_shape": (C.c_int, [_i32, _i32, _i32, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "ynb_load_conv": (C.c_int, [_p, _s, _p, _i64, _p, _i64]),
    "ynb_commit_weights": (C.c_int, [_p]),
    "ynb_forward_raw": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p]),
    "ynb_forward_decode": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p]),
    "ynb_forward_detect": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p]),
    "ynb_detect_host": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p]),
    "ynb_submit_host": (C.c_int, [_p, _i32, _p, _i32, _p, _p, _p, _p, _p]),
    "ynb_wait_host": (C.c_int, [_p, _i32]),
    "ynb_read_tap": (C.c_int, [_p, _s, _i32, _p, _p]),
    "ynb_tap_shape": (C.c_int, [_p, _s, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "ynb_launch_count": (_i64, [_p]),
    "ynb_set_profiling": (C.c_int, [_p, _i32]),
    "ynb_profile_count": (_i32, [_p]),
    "ynb_profile_entry": (C.c_int, [_p, _i32, C.POINTER(_s), C.POINTER(_s), C.POINTER(_f),
                                    C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ynb_dwconv3x3": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _i32, _p, _p,
                                _i32, _i32, _i32, _i32, _i32, _i32, _p]),
    "ynb_pwconv": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _i32, _p, _p,
                             _i64, _i32, _i32, _i32, _p]),
    "ynb_pwconv_tc": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _i32, _p, _p,
                                _i64, _i32, _i32, _i32, _i32, _p]),
    "ynb_dwpw_tc": (C.c_int, [_p, _i32, _p, _p, _i32, _p, _p, _i32, _p, _i32, _p, _i32,
                              _i32, _i32, _i32, _i32, _i32, _i32, _p]),
    "ynb_stem_pool": (C.c_int, [_p, _p, _p, _p, _i32, _i32, _p]),
    "ynb_decode_level": (C.c_int, [_p, _i32, _p, _p, _p, _i32, _i32, _i32, _i32,
                                   C.POINTER(_f), _i32, _i32, _i64, _i64, _p]),
    "ynb_nms_workspace_bytes": (_i64, [_i32, _i64]),
    "ynb_nms": (C.c_int, [_p, _p, _p, _i32, _i64, _i32, _f, _f, _i32,
                          _p, _p, _p, _p, _p, _p, _i64, _p]),
    "ynb_resize_bilinear": (C.c_int, [_p, _i32, _i32, _i32, _p, _i32, _i32, _p]),
    "ynb_set_normalization": (C.c_int, [_p, C.POINTER(_f), C.POINTER(_f)]),
    "ynb_preprocess_u8": (C.c_int, [_p, _p, _p, _i32, _p, _p]),
    "ynb_preprocess_letterbox_u8": (C.c_int, [_p, _p, _p, _i32, _p, _p]),
    "ynb_map_boxes": (C.c_int, [_p, _p, _p, _i32, _i64, _p]),
    "ynb_voc_append": (C.c_int, [_p, _p, _p, _p, _i32, _i64, _i32, _i32, _p, _i64, _p, _p]),
    "ynb_voc_eval_workspace_bytes": (_i64, [_i64, _i32, _i64]),
    "ynb_voc_eval": (C.c_int, [_p, _i64, _i32, _i32, _p, _p, _p, _i64, C.c_double, _i32, _p, _p, _p, _p, _p, _i64,
                               _p]),
    "ynb_coco_append": (C.c_int, [_p, _p, _p, _p, _i32, _i64, _i32, _i32, _p, _i64, _p, _p]),
    "ynb_coco_eval_workspace_bytes": (_i64, [_i64, _i32, _i32, _i64]),
    "ynb_coco_eval": (C.c_int, [_p, _i64, _i32, _i32, _p, _p, _i32, _p, _p, _p, _p, _i64, C.POINTER(C.c_double),
                                C.POINTER(C.c_double), _p, _p, _p, _i64, _p]),
    "ynb_submit_host_u8": (C.c_int, [_p, _i32, _p, _p, _i32, _p, _p, _p, _p, _p]),
    "ynb_nms_grid_workspace_bytes": (_i64, [_i32, _i32]),
    "ynb_nms_grid": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _f, _f, _i32,
                               _p, _p, _p, _p, _p, _p, _i64, _p]),
    "ynb_build_targets": (C.c_int, [_p, _p, _i32, _i32, _i32, C.POINTER(_f), _i32, _p, _p]),
    "ynb_train_loss_workspace_bytes": (_i64, [_i32, _i32]),
    "ynb_train_loss": (C.c_int, [_p, _p, _p, _i32, _p, _i32, _i32, C.POINTER(_f), _i32, _i32, _p, _p, _p, _p,
                                 _p, _i64, _p]),
    "ynb_raw_ld": (_i32, [_p]),
    "ynb_forward_train_loss": (C.c_int, [_p, _p, _i32, _p, _p, _p, _p, _p, _p, _i64, _p]),
    "ynb_sgd_step": (C.c_int, [_p, _p, _p, _i64, _f, _f, _f, _i32, _f, _p]),
    "ynb_dwconv3x3_bwd_data": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _i32, _i32, _i32, _i32, _i32, _p]),
    "ynb_dwconv3x3_bwd_weight_workspace_bytes": (_i64, [_i32, _i32, _i32, _i32, _i32]),
    "ynb_dwconv3x3_bwd_weight": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _i32, _i32, _i32, _i32, _i32,
                                           _p, _i64, _p]),
    "ynb_pwconv_bwd_weight_workspace_bytes": (_i64, [_i64, _i32, _i32]),
    "ynb_pwconv_bwd_weight": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _p, _i64, _i32, _i32, _p, _i64, _p]),
    "ynb_bn_workspace_bytes": (_i64, [_i64, _i32]),
    "ynb_bn_train_fwd": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _p, _p, _p, _p, _p, _i64, _i32, _f, _f, _i32,
                                   _p, _i64, _p]),
    "ynb_bn_train_bwd": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _i32, _i32, _p, _p, _p, _p, _i32, _i32, _p,
                                   _i64, _i32, _i32, _p, _i64, _p]),
    "ynb_conv3x3_bwd_weight": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _p, _i32, _i32, _i32, _i32, _i32, _p, _i64, _p]),
    "ynb_stem_conv_fwd": (C.c_int, [_p, _p, _p, _i32, _i32, _p]),
    "ynb_stem_conv_bwd_weight_workspace_bytes": (_i64, [_i32, _i32]),
    "ynb_stem_conv_bwd_weight": (C.c_int, [_p, _p, _p, _i32, _i32, _p, _i64, _p]),
    "ynb_maxpool3x3s2_fwd": (C.c_int, [_p, _p, _i32, _i32, _i32, _i32, _p]),
    "ynb_maxpool3x3s2_bwd": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _i32, _p]),
    "ynb_shuffle_unit_move": (C.c_int, [_p, _p, _p, _i64, _i32, _i32, _i32, _p]),
    "ynb_maxpool3x3s2_fwd_idx": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _i32, _p]),
    "ynb_maxpool3x3s2_bwd_idx": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _i32, _p]),
    "ynb_resample_add": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _i32, _i32, _p]),
    "ynb_resample_bwd": (C.c_int, [_p, _p, _i32, _i32, _i32, _i32, _i32, _p]),
    "ynb_add": (C.c_int, [_p, _p, _p, _i64, _p]),
    "ynb_conv3x3_tc": (C.c_int, [_p, _i32, _p, _i32, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p]),
    "ynb_tc_async_workspace_bytes": (C.c_int64, [_i32, _i32]),
    "ynb_pwconv_tc_async": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _i32, _p, _i32, _i32, _i32, _i32, _p, _i64, _i32, _i32,
                                      _i32, _i32, _p, _i64, _p]),
    "ynb_conv3x3_tc_async": (C.c_int, [_p, _i32, _p, _i32, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _i64, _p]),
    "ynb_ema_chunk_elems": (_i32, []),
    "ynb_ema_update": (C.c_int, [_p, _p, _p, _p, _p, _i32, _f, _f, _p]),
    "ynb_act_bwd": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _p, _i32, _i32, _i64, _i32, _i32, _p]),
}

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library and bind every declared symbol (raises if absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m yolo_nano_b200.build` "
            "(there is no CPU / PyTorch fallback for this path)")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.ynb_abi_version() != YNB_ABI_VERSION:
        raise ImportError("libyolonano_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib
