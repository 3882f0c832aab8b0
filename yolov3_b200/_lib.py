"""ctypes binding of include/yolov3_b200.h.  There is NO fallback: if the shared library is missing, or a call
fails, this raises — the product path never routes around the CUDA extension."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "libyolov3_b200.so"
_lib = None


class Y3Error(RuntimeError):
    pass


class ConvDesc(C.Structure):
    """struct y3_conv_desc (include/yolov3_b200.h)."""

    _fields_ = [
        ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
        ("c_in", C.c_int32), ("c_out", C.c_int32),
        ("ksize", C.c_int32), ("stride", C.c_int32),
        ("act", C.c_int32),
        ("in_", C.c_void_p), ("in_ld", C.c_int32), ("in_coff", C.c_int32),
        ("weight", C.c_void_p),
        ("bias", C.c_void_p),
        ("out", C.c_void_p), ("out_ld", C.c_int32), ("out_coff", C.c_int32),
        ("res", C.c_void_p), ("res_ld", C.c_int32), ("res_coff", C.c_int32),
        ("upsample", C.c_int32),
        ("out_f32", C.c_void_p), ("out_f32_ld", C.c_int32),
        ("err", C.c_void_p),
        ("weight_layout", C.c_int32),
    ]


class ConvPlanInfo(C.Structure):
    """struct y3_conv_plan_info."""

    _fields_ = [(k, C.c_int32) for k in ("block_n", "block_k", "pair", "staged", "halo", "resident_weights", "epilogue_groups",
                                         "xpair", "m_tiles", "n_tiles", "k_blocks", "grid")]


W_TAPS, W_XPAIR = 0, 1
MAX_LEVELS, MAX_ANCHORS = 5, 6


class DetectLevel(C.Structure):
    """struct y3_detect_level."""

    _fields_ = [("raw", C.c_void_p), ("head", C.c_void_p), ("head_ld", C.c_int32), ("raw_out", C.c_void_p),
                ("ny", C.c_int32), ("nx", C.c_int32), ("stride", C.c_float),
                ("anchor_w", C.c_float * MAX_ANCHORS), ("anchor_h", C.c_float * MAX_ANCHORS)]


class FirstDesc(C.Structure):
    """struct y3_first_desc."""

    _fields_ = [("in_", C.c_void_p), ("in_dtype", C.c_int32), ("in_div", C.c_float),
                ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("weight", C.c_void_p), ("bias", C.c_void_p), ("c_out", C.c_int32),
                ("out", C.c_void_p), ("out_ld", C.c_int32), ("out_coff", C.c_int32)]


class PoolDesc(C.Structure):
    """struct y3_pool_desc."""

    _fields_ = [("in_", C.c_void_p), ("in_ld", C.c_int32), ("in_coff", C.c_int32),
                ("out", C.c_void_p), ("out_ld", C.c_int32), ("out_coff", C.c_int32),
                ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c", C.c_int32),
                ("ho", C.c_int32), ("wo", C.c_int32),
                ("k", C.c_int32), ("stride", C.c_int32), ("off", C.c_int32), ("oob_zero", C.c_int32)]


class DecodeDesc(C.Structure):
    """struct y3_decode_desc."""

    _fields_ = [("levels", DetectLevel * MAX_LEVELS), ("nl", C.c_int32), ("bs", C.c_int32), ("na", C.c_int32),
                ("no", C.c_int32), ("z", C.c_void_p)]


OP_CONV_FIRST, OP_CONV, OP_MAXPOOL, OP_DECODE = 1, 2, 3, 4
IN_F32, IN_U8 = 0, 1


class Op(C.Structure):
    """struct y3_op."""

    _fields_ = [("kind", C.c_int32), ("conv", ConvDesc), ("first", FirstDesc), ("pool", PoolDesc),
                ("decode", DecodeDesc)]


class NmsParams(C.Structure):
    """struct y3_nms_params."""

    _fields_ = [("bs", C.c_int32), ("n_rows", C.c_int32), ("nc", C.c_int32),
                ("conf_thres", C.c_float), ("iou_thres", C.c_float),
                ("multi_label", C.c_int32), ("agnostic", C.c_int32),
                ("max_det", C.c_int32), ("max_nms", C.c_int32), ("max_wh", C.c_float),
                ("cap", C.c_int32), ("classes", C.POINTER(C.c_int32)), ("n_classes", C.c_int32)]


class LossDesc(C.Structure):
    """struct y3_loss_desc."""

    _fields_ = [("nl", C.c_int32), ("bs", C.c_int32), ("na", C.c_int32), ("nc", C.c_int32),
                ("p", C.c_void_p * MAX_LEVELS), ("grad", C.c_void_p * MAX_LEVELS),
                ("ny", C.c_int32 * MAX_LEVELS), ("nx", C.c_int32 * MAX_LEVELS),
                ("anchors", ((C.c_float * 2) * MAX_ANCHORS) * MAX_LEVELS),
                ("targets", C.c_void_p), ("nt", C.c_int32),
                ("box", C.c_float), ("obj", C.c_float), ("cls", C.c_float),
                ("cls_pw", C.c_float), ("obj_pw", C.c_float), ("anchor_t", C.c_float),
                ("cp", C.c_float), ("cn", C.c_float),
                ("balance", C.c_float * MAX_LEVELS), ("grad_scale", C.c_float)]


class BnActDesc(C.Structure):
    """struct y3_bn_act_desc."""

    _fields_ = [("y", C.c_void_p), ("y_ld", C.c_int32), ("y_coff", C.c_int32),
                ("res", C.c_void_p), ("res_ld", C.c_int32), ("res_coff", C.c_int32),
                ("out", C.c_void_p), ("out_ld", C.c_int32), ("out_coff", C.c_int32),
                ("scale", C.c_void_p), ("shift", C.c_void_p),
                ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c", C.c_int32), ("upsample", C.c_int32)]


class BnBwdDesc(C.Structure):
    """struct y3_bn_bwd_desc."""

    _fields_ = [("y", C.c_void_p), ("y_ld", C.c_int32), ("y_coff", C.c_int32),
                ("da", C.c_void_p), ("da_ld", C.c_int32), ("da_coff", C.c_int32),
                ("dy", C.c_void_p), ("dy_ld", C.c_int32), ("dy_coff", C.c_int32),
                ("scale", C.c_void_p), ("shift", C.c_void_p), ("mean", C.c_void_p), ("rstd", C.c_void_p),
                ("sums", C.c_void_p), ("partial", C.c_void_p), ("dbeta_acc", C.c_void_p), ("dgamma_acc", C.c_void_p),
                ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c", C.c_int32), ("upsample", C.c_int32),
                ("phase", C.c_int32), ("count", C.c_float)]


class WgradDesc(C.Structure):
    """struct y3_wgrad_desc."""

    _fields_ = [("dy", C.c_void_p), ("dy_ld", C.c_int32), ("dy_coff", C.c_int32),
                ("x", C.c_void_p), ("x_ld", C.c_int32), ("x_coff", C.c_int32),
                ("dw", C.c_void_p),
                ("co", C.c_int32), ("ci", C.c_int32), ("ksize", C.c_int32), ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("dw_layout", C.c_int32), ("accumulate", C.c_int32), ("deterministic", C.c_int32), ("stride", C.c_int32)]


DW_OIHW, DW_TAP_MAJOR, DW_OHWI = 0, 1, 2


class LetterboxDesc(C.Structure):
    """struct y3_letterbox_desc."""

    _fields_ = [("src", C.c_void_p), ("src_h", C.c_int32), ("src_w", C.c_int32), ("src_pitch", C.c_int32),
                ("new_h", C.c_int32), ("new_w", C.c_int32), ("top", C.c_int32), ("left", C.c_int32),
                ("dst", C.c_void_p), ("out_h", C.c_int32), ("out_w", C.c_int32),
                ("out_chw", C.c_int32), ("swap_rb", C.c_int32), ("pad", C.c_uint8 * 4)]


class PackItem(C.Structure):
    """struct y3_pack_item."""

    _fields_ = [("src_off", C.c_int64), ("dst", C.c_void_p), ("co_rows", C.c_int32), ("ci", C.c_int32), ("k", C.c_int32),
                ("dst_co", C.c_int32), ("tile_begin", C.c_int32), ("reserved", C.c_int32)]


def _declare(lib):
    i32, vp, sz = C.c_int32, C.c_void_p, C.c_size_t
    sigs = {
        "y3_version": ([], C.c_int),
        "y3_last_error": ([C.c_char_p, sz], C.c_int),
        "y3_device_check": ([], C.c_int),
        "y3_conv_bn_act_fwd": ([C.POINTER(ConvDesc), vp], C.c_int),
        "y3_conv_dgrad_s2": ([C.POINTER(ConvDesc), vp], C.c_int),
        "y3_conv_cout_pad": ([i32], C.c_int),
        "y3_conv_weight_layout": ([C.POINTER(ConvDesc)], C.c_int),
        "y3_conv_plan": ([C.POINTER(ConvDesc), C.POINTER(ConvPlanInfo)], C.c_int),
        "y3_abi_sizeof": ([i32], C.c_int64),
        "y3_set_pdl": ([i32], C.c_int),
        "y3_set_bn_async": ([i32], C.c_int),
        "y3_conv_first_fwd": ([C.POINTER(FirstDesc), vp], C.c_int),
        "y3_maxpool_fwd": ([C.POINTER(PoolDesc), vp], C.c_int),
        "y3_maxpool_train_fwd": ([C.POINTER(PoolDesc), vp, vp], C.c_int),
        "y3_maxpool_bwd": ([C.POINTER(PoolDesc), vp, i32, vp], C.c_int),
        "y3_bn_partial_blocks": ([i32, i32, i32, i32], i32),
        "y3_bn_stats": ([vp, i32, i32, i32, i32, i32, i32, vp, vp], C.c_int),
        "y3_colreduce_f32": ([vp, i32, i32, vp, i32, vp], C.c_int),
        "y3_bn_finalize": ([vp, i32, vp, vp, i32, C.c_float, C.c_float, C.c_float, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "y3_f32_to_bf16": ([vp, vp, C.c_int64, vp], C.c_int),
        "y3_pack_dgrad_batched": ([vp, i32, vp, i32, vp], C.c_int),
        "y3_head_grad_pack": ([vp, i32, i32, i32, i32, i32, vp, i32, i32, vp, vp], C.c_int),
        "y3_letterbox_u8": ([C.POINTER(LetterboxDesc), vp], C.c_int),
        "y3_scale_img_f32": ([vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, C.c_float, vp, vp], C.c_int),
        "y3_tta_merge": ([vp, i32, i32, i32, i32, i32, C.c_float, i32, C.c_float, vp, i32, i32, vp], C.c_int),
        "y3_val_match": ([vp, vp, i32, i32, i32, vp, i32, vp, i32, C.c_float, vp, vp, vp], C.c_int),
        "y3_ap_per_class_workspace_bytes": ([C.c_int64, C.c_int64, i32, i32], C.c_int64),
        "y3_ap_per_class": ([vp, C.c_int64, vp, C.c_int64, vp, i32, C.c_int64, vp, C.c_int64, vp, C.c_int64, C.c_int64, i32,
                             C.c_double, vp, C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp], C.c_int),
        "y3_confusion_update": ([vp, vp, i32, i32, i32, vp, i32, i32, C.c_float, C.c_float, C.c_float, vp, vp, vp], C.c_int),
        "y3_sumsq_blocks": ([], i32),
        "y3_grad_sumsq": ([vp, C.c_int64, vp, vp, vp], C.c_int),
        "y3_sgd_step": ([vp, vp, vp, vp, vp, C.c_int64, vp, vp, vp], C.c_int),
        "y3_bn_act_fwd": ([C.POINTER(BnActDesc), vp], C.c_int),
        "y3_bn_act_bwd": ([C.POINTER(BnBwdDesc), vp], C.c_int),
        "y3_pack_weights": ([vp, i32, i32, i32, vp, vp, vp], C.c_int),
        "y3_zero_stuff": ([vp, i32, i32, vp, i32, i32, i32, i32, i32, i32, vp], C.c_int),
        "y3_scale_boxes": ([vp, C.c_int64, i32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, vp], C.c_int),
        "y3_conv_wgrad": ([C.POINTER(WgradDesc), vp], C.c_int),
        "y3_conv_wgrad_tap_major": ([i32], C.c_int),
        "y3_conv_wgrad_s2_supported": ([i32, i32], C.c_int),
        "y3_add_nhwc": ([vp, i32, i32, vp, i32, i32, i32, i32, i32, i32, i32, vp], C.c_int),
        "y3_im2col_first": ([vp, i32, C.c_float, i32, i32, i32, vp, i32, i32, vp], C.c_int),
        "y3_colsum_f32": ([vp, i32, i32, C.c_int64, vp, vp], C.c_int),
        "y3_box_iou": ([vp, i32, vp, i32, C.c_float, vp, vp], C.c_int),
        "y3_loss_workspace_bytes": ([C.POINTER(LossDesc)], C.c_int64),
        "y3_loss_fwd_bwd": ([C.POINTER(LossDesc), vp, C.c_int64, vp, vp], C.c_int),
        "y3_model_create": ([C.POINTER(Op), i32, C.POINTER(vp)], C.c_int),
        "y3_model_forward": ([vp, vp, vp], C.c_int),
        "y3_model_num_launches": ([vp], i32),
        "y3_model_forward_timed": ([vp, vp, vp, C.POINTER(C.c_float), i32], C.c_int),
        "y3_model_destroy": ([vp], None),
        "y3_nchw_to_padded_nhwc": ([vp, i32, i32, i32, i32, vp, i32, i32, vp], C.c_int),
        "y3_padded_nhwc_to_nchw": ([vp, i32, i32, i32, i32, i32, i32, vp, vp], C.c_int),
        "y3_detect_decode_fwd": ([C.POINTER(DetectLevel), i32, i32, i32, i32, vp, vp], C.c_int),
        "y3_detect_head_decode_fwd": ([C.POINTER(DecodeDesc), vp], C.c_int),
        "y3_nms_default_capacity": ([i32, i32, i32], i32),
        "y3_nms_workspace_bytes": ([i32, i32], C.c_int64),
        "y3_nms_batched": ([vp, C.POINTER(NmsParams), vp, C.c_int64, vp, vp, vp, vp, vp], C.c_int),
    }
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    return sigs


SYMBOLS: dict = {}


def lib():
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise Y3Error(
                f"{_LIB_PATH} is missing: build it with `python -m yolov3_b200.build` (or __graft_entry__.build()). "
                "yolov3_b200 has no CPU or PyTorch fallback path."
            )
        _lib = C.CDLL(str(_LIB_PATH))
        SYMBOLS.update(_declare(_lib))
        for which, st in enumerate((ConvDesc, FirstDesc, PoolDesc, DetectLevel, DecodeDesc, Op, NmsParams, LossDesc, BnActDesc,
                                    BnBwdDesc, WgradDesc, PackItem, LetterboxDesc)):
            if _lib.y3_abi_sizeof(which) != C.sizeof(st):
                raise Y3Error(f"ABI mismatch: sizeof({st.__name__}) is {C.sizeof(st)} here, "
                              f"{_lib.y3_abi_sizeof(which)} in {_LIB_PATH.name}; rebuild the library")
    return _lib


def last_error() -> str:
    buf = C.create_string_buffer(1024)
    lib().y3_last_error(buf, 1024)
    return buf.value.decode(errors="replace")


def check(rc: int, what: str = ""):
    if rc != 0:
        raise Y3Error(f"{what or 'yolov3_b200'} failed (rc={rc}): {last_error()}")
