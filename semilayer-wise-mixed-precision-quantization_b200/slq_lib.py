"""slq_lib.py -- ctypes binding of libslq_b200.so (include/slq.h).

This is the ONLY way the Python host reaches the CUDA kernels: plain pointers and sizes across a
C ABI; torch only provides device memory (``tensor.data_ptr()``) and the current CUDA stream.
There is no CPU fallback: if the library cannot be loaded, every entry point raises.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libslq_b200.so")

SLQ_OK, SLQ_ERR_INVALID, SLQ_ERR_CUDA, SLQ_ERR_ZERO_RANGE, SLQ_ERR_UNSUPPORTED = 0, 1, 2, 3, 4
ROW_OK, ROW_ZERO_RANGE, ROW_CODE_RANGE = 0, 1, 2
DIV_TRUE, DIV_RECIP = 0, 1
IMPL_UMMA, IMPL_SIMT = 0, 1
A_AUTO, A_IM2COL, A_TILED = 0, 1, 2
OUT_U8, OUT_F32, OUT_ACC, OUT_S8 = 0, 1, 2, 3
IN_F32, IN_F16, IN_U8 = 0, 1, 2  # element type of the image handed to the stem (slq_stem_launch_in)
CALIB_PERCENTILE, CALIB_MSE, CALIB_ENTROPY = 1, 2, 3  # threshold rule of slq_hist_scales

_i32, _i64, _vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, _i32) for n in
                ("N", "H", "W", "Cin", "Cout", "kh", "kw", "stride", "pad", "w16", "impl", "a_mode")]


class Epilogue(ctypes.Structure):
    _fields_ = [("wscale", _vp), ("zf", _vp), ("bias", _vp), ("act_scales", _vp),
                ("in_id", _i32), ("out_id", _i32), ("res_id", _i32),
                ("res", _vp), ("res_signed", _i32),
                ("out", _vp), ("out_S", _vp), ("out_mode", _i32), ("relu", _i32),
                ("in_rowsum", _vp), ("out_rowsum", _vp), ("in_planes", _i32), ("in_plane_stride", _i64)]


class BlockTailDesc(ctypes.Structure):
    _fields_ = [(n, _i32) for n in ("N", "H", "W", "Cin", "stride", "Cmid", "Cout", "impl")]


class BlockTailEpilogue(ctypes.Structure):
    _fields_ = [("wscale3", _vp), ("zf3", _vp), ("bias3", _vp), ("wscaled", _vp), ("zfd", _vp), ("biasd", _vp),
                ("act_scales", _vp), ("in3_id", _i32), ("ind_id", _i32), ("out_id", _i32),
                ("out", _vp), ("out_mode", _i32), ("out_rowsum", _vp)]


# name -> (restype, argtypes); mirrors include/slq.h one to one (tests check the export list)
SIGNATURES = {
    "slq_last_error": (ctypes.c_char_p, []),
    "slq_abi_version": (ctypes.c_int, []),
    "slq_device_info": (ctypes.c_int, [_vp, _vp, _vp]),
    "slq_packed_row_bytes": (_i64, [_i64, _i32]),
    "slq_quantize_rows": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "slq_quantize_rows_host": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "slq_quantize_jobs": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "slq_decode_rows": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp]),
    "slq_eval_tail": (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "slq_kl_rows": (ctypes.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "slq_probe_i8_peak": (ctypes.c_int, [_i32, ctypes.POINTER(_i64), _vp]),
    "slq_classify_rows": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "slq_encode_rows": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "slq_gemm_weight_rows": (_i64, [ctypes.POINTER(ConvDesc)]),
    "slq_build_gemm_weights": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp]),
    "slq_conv_create": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, ctypes.POINTER(_vp)]),
    "slq_conv_destroy": (None, [_vp]),
    "slq_conv_tiling": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp]),
    "slq_build_packed_gemm_weights": (ctypes.c_int, [ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "slq_conv_set_packed_weights": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "slq_conv_launch": (ctypes.c_int, [_vp, ctypes.POINTER(Epilogue), _vp]),
    "slq_blocktail_create": (ctypes.c_int, [ctypes.POINTER(BlockTailDesc), _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "slq_blocktail_destroy": (None, [_vp]),
    "slq_blocktail_rowsum_planes": (_i32, [_vp]),
    "slq_blocktail_launch": (ctypes.c_int, [_vp, ctypes.POINTER(BlockTailEpilogue), _vp]),
    "slq_debug_set_trace": (ctypes.c_int, [_vp, _i32]),
    "slq_stem_forward": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _vp, _vp]),
    "slq_conv_rowsum_planes": (_i32, [_vp, _i32]),
    "slq_conv_needs_rowsum": (_i32, [_vp, _i32]),
    "slq_stem_workspace_bytes": (_i64, [_i32, _i32, _i32]),
    "slq_stem_create": (ctypes.c_int, [_i32, _i32, _i32, _vp, ctypes.POINTER(_vp)]),
    "slq_stem_destroy": (None, [_vp]),
    "slq_stem_set_weights": (ctypes.c_int, [_vp, _vp, _vp]),
    "slq_stem_launch": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _vp]),
    "slq_stem_launch_in": (ctypes.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _vp]),
    "slq_tail_workspace_bytes": (_i64, [_i32, _i32, _i32]),
    "slq_tail_split_weights": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp]),
    "slq_tail_forward": (ctypes.c_int, [_vp, _i32, _i32, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "slq_absmax_scale": (ctypes.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp]),
    "slq_quantize_act": (ctypes.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp]),
    "slq_act_histogram": (ctypes.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp]),
    "slq_hist_scales": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _i32, ctypes.c_double, ctypes.c_float, _vp, _vp]),
}

_lib = None


class SlqError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libslq_b200: error %d: %s" % (code, msg))
        self.code = code


def lib():
    """Loads libslq_b200.so (building is __graft_entry__.build()'s / slq_build.build()'s job).
    $SLQ_DEBUG_LIB=1 loads the tracing build libslq_b200_dbg.so instead (developer tools only)."""
    global _lib, LIB_PATH
    if _lib is None:
        if os.environ.get("SLQ_DEBUG_LIB") == "1":
            import slq_build
            LIB_PATH = slq_build.build(debug=True)
        elif os.environ.get("SLQ_LIB_VARIANT"):  # developer tools: an A/B build of the same sources (tools/layer_time.py)
            LIB_PATH = os.path.join(HERE, "libslq_b200_%s.so" % os.environ["SLQ_LIB_VARIANT"])
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libslq_b200.so is missing (%s). Build it with `python slq_build.py`; this package "
                "has no CPU or eager-PyTorch fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.slq_abi_version() != 1:
            raise RuntimeError("libslq_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    if rc != SLQ_OK:
        msg = lib().slq_last_error()
        raise SlqError(rc, msg.decode() if msg else "")


def ptr(t):
    """Device/host address of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream(device=None):
    import torch
    return torch.cuda.current_stream(device).cuda_stream
