"""ctypes binding of libyre.so (the C ABI declared in include/yre.h).

There is no fallback: if the library is missing or the device is not a B200 the import of the
compute path fails loudly (north_star: "no Triton, no cuDNN/cuBLAS dispatch and no CPU fallback").
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libyre.so"

BF16, F32, F16 = 0, 1, 2
ACT_NONE, ACT_SILU = 0, 1
NHWC, PHASE4 = 0, 1
ENGINE_AUTO, ENGINE_FFMA, ENGINE_TCGEN05 = 0, 1, 2


class View(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("dtype", C.c_int32), ("layout", C.c_int32), ("B", C.c_int32), ("H", C.c_int32),
                ("W", C.c_int32), ("C_total", C.c_int32), ("c_off", C.c_int32), ("C", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [("x", View), ("y", View), ("res", View), ("w", C.c_void_p), ("bias", C.c_void_p),
                ("k", C.c_int32), ("stride", C.c_int32), ("act", C.c_int32), ("engine", C.c_int32), ("xu", View)]


TC_GENERIC, TC_GENERIC_CTA2, TC_HALO_WS, TC_HALO_STREAM = 0, 1, 2, 3


class TcSchedule(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("kind", "ybx", "tw", "th", "tb", "block_n", "tiles_x", "tiles_y", "tiles_b", "tiles_n",
                                         "mtiles", "npair", "upn", "work", "grid")]


class StemDesc(C.Structure):
    _fields_ = [("x_nchw", C.c_void_p), ("B", C.c_int32), ("Cin", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("y", View), ("w", C.c_void_p), ("bias", C.c_void_p), ("stride", C.c_int32), ("act", C.c_int32),
                ("x_u8_hwc", C.c_void_p)]


class DecodeDesc(C.Structure):
    _fields_ = [("raw", View * 8), ("stride", C.c_float * 8), ("levels", C.c_int32), ("nc", C.c_int32),
                ("dfl_w", C.c_float * 16), ("y", C.c_void_p)]


class DecodeMasksDesc(C.Structure):
    _fields_ = [("dec", DecodeDesc), ("mask", View * 8), ("nm", C.c_int32), ("mc", C.c_void_p)]


class NmsDesc(C.Structure):
    _fields_ = [("pred", C.c_void_p), ("B", C.c_int32), ("A", C.c_int32), ("nc", C.c_int32),
                ("conf_thres", C.c_float), ("iou_thres", C.c_double), ("max_det", C.c_int32),
                ("classes", C.c_void_p), ("n_classes", C.c_int32), ("agnostic", C.c_int32),
                ("out", C.c_void_p), ("counts", C.c_void_p), ("keep_anchor", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t), ("scale", C.c_void_p)]


class LetterboxDesc(C.Structure):
    _fields_ = [("src", C.c_void_p), ("h", C.c_int32), ("w", C.c_int32), ("row_pitch", C.c_int64),
                ("new_shape", C.c_int32), ("new_w", C.c_int32), ("new_h", C.c_int32), ("top", C.c_int32),
                ("left", C.c_int32), ("color", C.c_uint8 * 4), ("out_mode", C.c_int32), ("dst", C.c_void_p),
                ("out_h", C.c_int32), ("out_w", C.c_int32)]


LB_F32_CHW, LB_U8_HWC = 0, 1
YUV_NV12, YUV_NV21, YUV_I420, YUV_YV12 = 0, 1, 2, 3
YUV_BT601, YUV_BT709 = 0, 1


class Yuv420Planes(C.Structure):
    _fields_ = [("luma", C.c_void_p), ("luma_pitch", C.c_int64), ("chroma", C.c_void_p * 2), ("chroma_pitch", C.c_int64),
                ("format", C.c_int32), ("matrix", C.c_int32)]


class MatchDesc(C.Structure):
    _fields_ = [("det", C.c_void_p), ("det_stride", C.c_int32), ("det_off", C.c_void_p), ("gt_boxes", C.c_void_p),
                ("gt_cls", C.c_void_p), ("gt_off", C.c_void_p), ("B", C.c_int32), ("n_thr", C.c_int32), ("thr", C.c_double * 16),
                ("max_gt_per_image", C.c_int32), ("tp", C.c_void_p)]


TTA_BRANCHES = 3


class TtaGeom(C.Structure):
    _fields_ = [("h", C.c_int32), ("w", C.c_int32), ("scale", C.c_float * TTA_BRANCHES), ("flip", C.c_int32 * TTA_BRANCHES)] + \
               [(n, C.c_int32 * TTA_BRANCHES) for n in ("rh", "rw", "out_h", "out_w", "A", "a_begin", "a_end")] + [("A_tot", C.c_int32)]


class TtaScaleDesc(C.Structure):
    _fields_ = [("x_nchw", C.c_void_p), ("x_u8_hwc", C.c_void_p)] + \
               [(n, C.c_int32) for n in ("B", "n", "H", "W", "flip", "rh", "rw", "out_h", "out_w")] + [("y", C.c_void_p)]


class TtaMergeBranch(C.Structure):
    _fields_ = [("y", C.c_void_p), ("A", C.c_int32), ("a_begin", C.c_int32), ("a_end", C.c_int32), ("scale", C.c_float),
                ("flip_w", C.c_int32)]


class TtaMergeDesc(C.Structure):
    _fields_ = [("br", TtaMergeBranch * TTA_BRANCHES), ("B", C.c_int32), ("n", C.c_int32), ("nc", C.c_int32), ("out", C.c_void_p)]

MASK_PROTO, MASK_INPUT, MASK_NATIVE = 0, 1, 2


class MaskDesc(C.Structure):
    _fields_ = [("proto", C.c_void_p)] + [(n, C.c_int32) for n in ("B", "n", "mh", "mw", "nm", "proto_pitch")] + \
               [("mc", C.c_void_p), ("A", C.c_int32), ("det", C.c_void_p), ("counts", C.c_void_p), ("keep_anchor", C.c_void_p),
                ("max_det", C.c_int32), ("mode", C.c_int32), ("in_h", C.c_int32), ("in_w", C.c_int32), ("scale", C.c_void_p),
                ("masks", C.c_void_p), ("out_h", C.c_int32), ("out_w", C.c_int32)]


# name -> (restype, argtypes); every symbol include/yre.h declares
SYMBOLS = {
    "yre_version": (C.c_int, []),
    "yre_last_error": (C.c_char_p, []),
    "yre_device_check": (C.c_int, []),
    "yre_conv": (C.c_int, [C.POINTER(ConvDesc), C.c_void_p]),
    "yre_conv_tc_describe": (C.c_int, [C.POINTER(ConvDesc), C.c_int32, C.c_char_p, C.c_int32]),
    "yre_conv_tc_schedule": (C.c_int, [C.POINTER(ConvDesc), C.c_int32, C.c_int32, C.POINTER(TcSchedule)]),
    "yre_stem_conv": (C.c_int, [C.POINTER(StemDesc), C.c_void_p]),
    "yre_adown_prepool": (C.c_int, [C.POINTER(View)] * 3 + [C.c_void_p]),
    "yre_spp_maxpool": (C.c_int, [C.POINTER(View)] * 4 + [C.c_void_p]),
    "yre_upsample2x": (C.c_int, [C.POINTER(View)] * 2 + [C.c_void_p]),
    "yre_cbfuse_sum": (C.c_int, [C.POINTER(View), C.c_int32, C.POINTER(View), C.POINTER(View), C.c_void_p]),
    "yre_nchw_to_view": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_void_p]),
    "yre_view_to_nchw": (C.c_int, [C.POINTER(View), C.c_void_p, C.c_void_p]),
    "yre_dfl_decode_score": (C.c_int, [C.POINTER(DecodeDesc), C.c_void_p]),
    "yre_dfl_decode_score_masks": (C.c_int, [C.POINTER(DecodeMasksDesc), C.c_void_p]),
    "yre_nms_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32]),
    "yre_nms_batched": (C.c_int, [C.POINTER(NmsDesc), C.c_void_p]),
    "yre_nms_filter_only": (C.c_int, [C.POINTER(NmsDesc), C.c_void_p]),
    "yre_nms_multi_label_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32]),
    "yre_nms_batched_multi_label": (C.c_int, [C.POINTER(NmsDesc), C.c_void_p]),
    "yre_nms_multi_label_filter_only": (C.c_int, [C.POINTER(NmsDesc), C.c_void_p]),
    "yre_letterbox_geometry_rect": (C.c_int, [C.POINTER(LetterboxDesc), C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_double),
                                    C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "yre_letterbox_geometry": (C.c_int, [C.POINTER(LetterboxDesc), C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "yre_letterbox_u8": (C.c_int, [C.POINTER(LetterboxDesc), C.c_void_p]),
    "yre_letterbox_u8_batch": (C.c_int, [C.POINTER(LetterboxDesc), C.c_int32, C.c_void_p]),
    "yre_letterbox_yuv420_batch": (C.c_int, [C.POINTER(LetterboxDesc), C.POINTER(Yuv420Planes), C.c_int32, C.c_void_p]),
    "yre_scale_boxes": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]),
    "yre_match_detections": (C.c_int, [C.POINTER(MatchDesc), C.c_void_p]),
    "yre_tta_geometry": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(TtaGeom)]),
    "yre_tta_scale_img": (C.c_int, [C.POINTER(TtaScaleDesc), C.c_void_p]),
    "yre_tta_merge": (C.c_int, [C.POINTER(TtaMergeDesc), C.c_void_p]),
    "yre_seg_masks": (C.c_int, [C.POINTER(MaskDesc), C.c_void_p]),
    "yre_plan_create": (C.c_int, [C.POINTER(C.c_void_p)]),
    "yre_plan_destroy": (None, [C.c_void_p]),
    "yre_plan_add_conv": (C.c_int, [C.c_void_p, C.POINTER(ConvDesc)]),
    "yre_plan_add_stem": (C.c_int, [C.c_void_p, C.POINTER(StemDesc)]),
    "yre_plan_add_adown_prepool": (C.c_int, [C.c_void_p] + [C.POINTER(View)] * 3),
    "yre_plan_add_spp_maxpool": (C.c_int, [C.c_void_p] + [C.POINTER(View)] * 4),
    "yre_plan_add_upsample2x": (C.c_int, [C.c_void_p] + [C.POINTER(View)] * 2),
    "yre_plan_add_cbfuse_sum": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_int32, C.POINTER(View), C.POINTER(View)]),
    "yre_plan_add_nchw_to_view": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(View)]),
    "yre_plan_add_view_to_nchw": (C.c_int, [C.c_void_p, C.POINTER(View), C.c_void_p]),
    "yre_plan_add_decode": (C.c_int, [C.c_void_p, C.POINTER(DecodeDesc)]),
    "yre_plan_add_decode_masks": (C.c_int, [C.c_void_p, C.POINTER(DecodeMasksDesc)]),
    "yre_plan_add_nms": (C.c_int, [C.c_void_p, C.POINTER(NmsDesc)]),
    "yre_plan_rebind": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "yre_plan_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "yre_plan_run_batch": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "yre_plan_batch_capacity": (C.c_int, [C.c_void_p]),
    "yre_plan_run_op": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "yre_plan_num_launches": (C.c_int, [C.c_void_p]),
    "yre_plan_num_ops": (C.c_int, [C.c_void_p]),
    "yre_plan_num_tcgen05": (C.c_int, [C.c_void_p]),
    "yre_plan_op_flops": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_int32]),
    "yre_plan_op_name": (C.c_char_p, [C.c_void_p, C.c_int32]),
    "yre_plan_op_variant": (C.c_int, [C.c_void_p, C.c_int32, C.c_char_p, C.c_int32]),
}

_lib = None


class YreError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Loads libyre.so once.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise YreError(f"{LIB_PATH} not found: build it with `python yolo-re_b200/build.py` "
                           "(there is no CPU / cuDNN fallback for this path)")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)      # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().yre_last_error().decode(errors="replace")
        raise YreError(f"libyre {what} failed ({code}): {msg}")
