"""ctypes binding of liborp_b200.so (include/orp_b200.h).

There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
The library is built in-tree by `python -m orientedreppoints_b200.build` (nvcc, sm_100a).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "liborp_b200.so")

ORP_NMS_EXACT64, ORP_NMS_COMPAT32 = 0, 1
ORP_UNION_NAN_KEEPS, ORP_UNION_GUARD, ORP_UNION_NAN_SUPPRESSES = 0, 1, 2
ORP_ORDER_INDEX_ASC, ORP_ORDER_SCORE_DESC = 0, 1
ORP_RESIZE_MAX_RATES = 8

_vp = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_d = ctypes.c_double


class NmsStats(ctypes.Structure):
    _fields_ = [("pairs_total", ctypes.c_int64), ("pairs_aabb", ctypes.c_int64),
                ("pairs_clipped", ctypes.c_int64), ("pairs_fp64", ctypes.c_int64),
                ("edges", ctypes.c_int64), ("suppressing", ctypes.c_int64), ("overflow", ctypes.c_int32),
                ("rounds", ctypes.c_int32), ("n", ctypes.c_int32)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class TcProblem(ctypes.Structure):
    _fields_ = [("x", _vp), ("N", _i), ("H", _i), ("W", _i), ("out", _vp), ("residual_bf16", _vp),
                ("residual_f32", _vp), ("offset", _vp), ("gn_stats", _vp), ("mask", _vp)]


class GnProblem(ctypes.Structure):
    _fields_ = [("x", _vp), ("N", _i), ("H", _i), ("W", _i), ("stats", _vp), ("up_src", _vp), ("y", _vp)]


# name -> (restype, argtypes); every symbol include/orp_b200.h declares
SIGNATURES = {
    "orp_last_error": (ctypes.c_char_p, []),
    "orp_version": (_i, []),
    "orp_compiled_sm": (_i, []),
    "orp_launch_count": (ctypes.c_int64, []),
    "orp_reset_launch_count": (None, []),
    "orp_rnms": (_i, [_vp, _vp, _i, _d, _i, _i, _i, _vp, _vp, _vp]),
    "orp_poly_nms_host": (_i, [_vp, _vp, _vp, _i, _i, _f, _i]),
    "orp_rnms_last_stats": (_i, [ctypes.POINTER(NmsStats)]),
    "orp_set_timing": (None, [_i]),
    "orp_rnms_last_sweep_ms": (_i, [ctypes.POINTER(ctypes.c_float)]),
    "orp_tc_timing_collect": (_i, [ctypes.POINTER(ctypes.c_float), ctypes.POINTER(_i), ctypes.POINTER(_d)]),
    "orp_poly_overlaps_host": (_i, [_vp, _vp, _vp, _i, _i, _i]),
    "orp_poly_overlaps": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "orp_quad_iou_matrix": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp]),
    "orp_iou_poly_f64_pairs": (_i, [_vp, _vp, _i, _vp, _vp]),
    "orp_box_iou_rotated": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "orp_minarearect": (_i, [_vp, _i, _vp, _vp, _f, _vp, _vp]),
    "orp_head_postprocess": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _d, _i, _vp, _vp, _vp, _vp, _vp]),
    "orp_pack_detections": (_i, [_vp, _vp, _vp, _i, _i, _vp, _vp]),
    "orp_dcn_offsets_multi": (_i, [_i, _vp, _vp, _vp, _f, _vp, _vp]),
    "orp_conv2d_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _i, _vp]),
    "orp_deform_conv2d_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "orp_gn_apply_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _f, _i, _vp, _vp, _vp]),
    "orp_maxpool3x3s2_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_conv2d_bf16": (_i, [_i, ctypes.POINTER(TcProblem), _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "orp_conv2d_f16x3": (_i, [_i, ctypes.POINTER(TcProblem), _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    "orp_conv2d_tc_splitk": (_i, [ctypes.POINTER(TcProblem), _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_f16x3_overflow_count": (_i, [ctypes.POINTER(ctypes.c_uint), _i]),
    "orp_stem_s2d_u8_f16x3": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orp_stem_s2d_f16x3": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_stem_conv_s2d_f16x3": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "orp_maxpool3x3s2_f16x3": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_gn_stats_f16x3": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_gn_apply_f16x3_multi": (_i, [_i, _vp, _i, _i, _vp, _vp, _f, _i, _vp]),
    "orp_split_from_f32": (_i, [_vp, ctypes.c_longlong, _i, _vp, _vp]),
    "orp_split_to_f32": (_i, [_vp, ctypes.c_longlong, _i, _vp, _vp]),
    "orp_transpose_f32": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_nchw_f32_to_split": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_layernorm_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _f, _i, _i, _vp, _vp]),
    "orp_window_attention_bf16": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _f, _vp, _vp]),
    "orp_patch_embed_rows_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_patch_embed_rows_u8_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orp_patch_merge_gather_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_subsample2_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_stem_conv_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orp_layernorm_f16x3": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _f, _i, _i, _vp, _vp]),
    "orp_window_attention_f16x3": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _f, _vp, _vp]),
    "orp_patch_embed_rows_f16x3": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_patch_embed_rows_u8_f16x3": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orp_patch_merge_gather_f16x3": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_subsample2_f16x3": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_stem_im2col_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_stem_s2d_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "orp_convex_iou": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "orp_split_tiles_u8": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _vp, _vp]),
    "orp_resize_cubic_table": (_i, [_i, _d, _i, _vp, _vp, _vp]),
    "orp_resize_tiles_cubic_u8": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "orp_resize_cubic_u8": (_i, [_vp, _i, _i, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp]),
    "orp_stem_s2d_u8_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orp_stem_conv_s2d_bf16": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "orp_maxpool3x3s2_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_gn_stats_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "orp_gn_apply_bf16": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _f, _i, _vp, _vp, _vp]),
    "orp_gn_apply_bf16_multi": (_i, [_i, _vp, _i, _i, _vp, _vp, _f, _i, _vp]),
}

_LIB = None


class OrpError(RuntimeError):
    pass


def lib():
    """Load the CUDA library; raises (never falls back) when it is absent."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise OrpError(
                "liborp_b200.so not found at %s - build it with `python -m orientedreppoints_b200.build` "
                "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)   # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _LIB = l
    return _LIB


def check(rc, what=""):
    if rc != 0:
        msg = lib().orp_last_error()
        raise OrpError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else ""))


def launch_count():
    return int(lib().orp_launch_count())


def reset_launch_count():
    lib().orp_reset_launch_count()


def last_nms_stats():
    s = NmsStats()
    check(lib().orp_rnms_last_stats(ctypes.byref(s)), "orp_rnms_last_stats")
    return s.as_dict()


def set_timing(on):
    lib().orp_set_timing(1 if on else 0)


def last_sweep_ms():
    v = ctypes.c_float(0)
    check(lib().orp_rnms_last_sweep_ms(ctypes.byref(v)), "orp_rnms_last_sweep_ms")
    return float(v.value)


def tc_timing_collect():
    ms, n, fl = ctypes.c_float(0), ctypes.c_int(0), ctypes.c_double(0)
    check(lib().orp_tc_timing_collect(ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl)), "orp_tc_timing_collect")
    return float(ms.value), int(n.value), float(fl.value)


def current_stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """device/host pointer of a torch tensor (None -> NULL)"""
    return ctypes.c_void_p(0 if t is None else t.data_ptr())
