"""ctypes binding of libss4k.so (include/ss4k.h).  No torch types cross this boundary."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libss4k.so")

OK = 0
ARCH_SRVGG, ARCH_RRDB, ARCH_BSVD = 0, 1, 2
DT_F32, DT_F16 = 0, 1
ACT_F16, ACT_BF16, ACT_F16_SPLIT = 0, 1, 2
FMT_F32_NCHW, FMT_F16_NCHW, FMT_U8_NHWC, FMT_NV12 = 0, 1, 2, 3
MODE_CONV3, MODE_UP2, MODE_S2 = 0, 1, 2


class PlanCfg(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "struct_size", "net_id", "arch", "n", "h", "w", "scale", "depth", "tile", "tile_pad",
        "act_mode", "in_fmt", "out_fmt", "use_graph")] + [("reserved", ctypes.c_int32 * 8)]


class Nv12Surface(ctypes.Structure):
    """ss4k_nv12_surface (include/ss4k.h): one pitched NV12 frame of a hardware decoder / encoder"""
    _fields_ = [("y", ctypes.c_void_p), ("uv", ctypes.c_void_p), ("pitch_y", ctypes.c_int32), ("pitch_uv", ctypes.c_int32)]


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "struct_size", "n", "h", "w", "cin", "cout", "mode", "act", "act_mode", "pixel_shuffle")] + [
        ("alpha", ctypes.c_float), ("beta", ctypes.c_float), ("reserved", ctypes.c_int32 * 8)]


# every symbol include/ss4k.h declares: name -> (restype, argtypes)
_vp, _i, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
SYMBOLS = {
    "ss4k_abi_version": (_i, []),
    "ss4k_create": (_i, [_i, ctypes.POINTER(_vp)]),
    "ss4k_destroy": (_i, [_vp]),
    "ss4k_last_error": (ctypes.c_char_p, [_vp]),
    "ss4k_desc_mode": (_i, [_vp]),
    "ss4k_set_desc_mode": (_i, [_vp, _i]),
    "ss4k_launch_count": (_i64, [_vp]),
    "ss4k_load_weights": (_i, [_vp, _i, ctypes.c_char_p, _vp, _i, ctypes.POINTER(_i64), _i]),
    "ss4k_clear_weights": (_i, [_vp, _i]),
    "ss4k_plan_create": (_i, [_vp, ctypes.POINTER(PlanCfg), ctypes.POINTER(_vp)]),
    "ss4k_plan_destroy": (_i, [_vp]),
    "ss4k_plan_out_shape": (_i, [_vp, ctypes.POINTER(ctypes.c_int32 * 4)]),
    "ss4k_plan_flops": (ctypes.c_double, [_vp]),
    "ss4k_plan_launches": (_i, [_vp]),
    "ss4k_plan_graph_steps": (_i, [_vp]),
    "ss4k_plan_steps": (_i, [_vp]),
    "ss4k_debug_tile_layout": (_i, [_vp, ctypes.POINTER(ctypes.c_void_p)]),
    "ss4k_debug_bsvd_stream_layout": (_i, [_vp, _i, ctypes.POINTER(ctypes.c_void_p)]),
    "ss4k_plan_dry": (_i, [ctypes.POINTER(PlanCfg), ctypes.POINTER(_vp)]),
    "ss4k_free": (None, [_vp]),
    "ss4k_run": (_i, [_vp, _vp, _vp, _vp]),
    "ss4k_run_host": (_i, [_vp, _vp, _vp]),
    "ss4k_run_host_async": (_i, [_vp, _vp, _vp]),
    "ss4k_plan_host_sync": (_i, [_vp]),
    "ss4k_plan_io_bytes": (_i, [_vp, ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    "ss4k_plan_profile": (_i, [_vp, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double),
                               ctypes.POINTER(ctypes.c_int32), _i]),
    "ss4k_bsvd_stream_open": (_i, [_vp, ctypes.POINTER(_vp)]),
    "ss4k_bsvd_stream_open_batched": (_i, [_vp, _i, ctypes.POINTER(_vp)]),
    "ss4k_bsvd_stream_push": (_i, [_vp, _vp, _vp, ctypes.POINTER(_i), _vp]),
    "ss4k_bsvd_stream_push_frames": (_i, [_vp, _vp, _i, _vp, ctypes.POINTER(_i), _vp]),
    "ss4k_bsvd_stream_flush": (_i, [_vp, _vp, ctypes.POINTER(_i), _vp]),
    "ss4k_bsvd_stream_reset": (_i, [_vp]),
    "ss4k_bsvd_stream_latency": (_i, [_vp]),
    "ss4k_bsvd_stream_close": (_i, [_vp]),
    "ss4k_rgb_to_nv12": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "ss4k_nv12_pack": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "ss4k_nv12_unpack": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "ss4k_glue_chan_stats": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "ss4k_glue_area_pool": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "ss4k_glue_blur_diff": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp]),
    "ss4k_glue_finalize": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp, _vp,
                                _i, _vp]),
    "ss4k_glue_finalize_bicubic_u8": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp,
                                           _i, _i, _i, _vp]),
    "ss4k_glue_finalize_nv12": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, ctypes.c_double, ctypes.c_double, _vp,
                                     _i, _vp]),
    "ss4k_glue_finalize_bicubic_nv12": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, ctypes.c_double, ctypes.c_double,
                                             _vp, _i, _i, _i, _vp]),
    "ss4k_glue_bicubic_u8": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "ss4k_glue_sharpen_blend": (_i, [_vp, _i, _i, _i, _i, _i, ctypes.c_float, ctypes.c_float, _vp, _i, _vp, _vp]),
    "ss4k_glue_sharpen_blend_act": (_i, [_vp, _i, _i, _i, _i, _i, ctypes.c_float, ctypes.c_float, _vp, _i, _vp, _i, _i, _i, _vp]),
    "ss4k_plan_input_act": (_i, [_vp, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int32),
                                ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "ss4k_run_act": (_i, [_vp, _vp, _vp]),
    "ss4k_conv3x3": (_i, [_vp, ctypes.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ss4k_debug_bench_conv": (_i, [_vp, ctypes.POINTER(ConvDesc), _i, _i, _i, ctypes.POINTER(ctypes.c_float),
                                   ctypes.POINTER(_vp)]),
    "ss4k_debug_pack": (_i, [ctypes.POINTER(ConvDesc), _i, _i, _i, _vp, _vp, _vp, ctypes.POINTER(_vp),
                             ctypes.POINTER(_vp), ctypes.POINTER(_i64)]),
}

_lib = None


class Ss4kError(RuntimeError):
    """Raised for every non-zero return of the C ABI (so BaseService.proc_main's ``except`` path,
    reference src/upscale/base_service.py:64-70, still fires)."""


def load():
    """Load libss4k.so; there is no fallback: a missing library is a hard error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise Ss4kError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). This engine has no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, ctx=None):
    if rc != OK:
        msg = load().ss4k_last_error(ctx)
        raise Ss4kError(f"ss4k error {rc}: {msg.decode() if msg else '?'}")
