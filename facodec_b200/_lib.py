"""ctypes binding of include/facodec_b200.h (the C-ABI shared library built by
facodec_b200/build.py).  There is NO fallback: if the library is missing or a
call fails, an exception is raised -- the product never routes through a CPU path."""
import ctypes
import os

from . import build as _build

_c = ctypes
_LIB = None


class FacError(RuntimeError):
    pass


def lib_path():
    return _build.LIB


def load():
    """Loads facodec_b200/_C/libfacodec_b200.so (built in-tree by `python -m facodec_b200.build`)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise FacError(f"{path} not found: build it with `python -m facodec_b200.build` "
                       "(needs nvcc; there is no CPU fallback)")
    L = ctypes.CDLL(path)
    vp, i32, i64p, fp = _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p
    sigs = {
        "fac_abi_version": ([], i32),
        "fac_create": ([_c.POINTER(vp), i32], i32),
        "fac_destroy": ([vp], i32),
        "fac_last_error": ([vp], _c.c_char_p),
        "fac_load_tensor": ([vp, i32, _c.c_char_p, fp, _c.POINTER(_c.c_int64), i32], i32),
        "fac_finalize": ([vp], i32),
        "fac_encode": ([vp, fp, i32, i32, fp, vp], i32),
        "fac_encode_frames": ([i32], i32),
        "fac_quantize": ([vp, fp, fp, i32, i32, i32, i32, fp, i32, i64p, fp, fp, fp, fp, fp, fp, i64p, i64p, i64p, vp], i32),
        "fac_decode": ([vp, fp, i32, i32, fp, vp], i32),
        "fac_codec_forward": ([vp, fp, i32, i32, i32, fp, i64p, i64p, i64p, fp, vp], i32),
        "fac_codec_forward_host": ([vp, fp, i32, i32, i32, fp, i64p, i64p, i64p, vp], i32),
        "fac_redecode": ([vp, i64p, i64p, i32, fp, i32, i32, i32, i32, i32, fp, vp], i32),
        "fac_redecoder_decode": ([vp, fp, i32, i32, fp, vp], i32),
        "fac_voice_convert": ([vp, i64p, i64p, i32, fp, i32, i32, i32, i32, i32, fp, vp], i32),
        "fac_dequantize": ([vp, i64p, i64p, i32, i32, i64p, i32, i32, fp, i32, i32, fp, fp, fp, fp, vp], i32),
        "fac_decode_codes": ([vp, i64p, i64p, i32, i32, i64p, i32, i32, fp, i32, i32, fp, vp], i32),
        "fac_dataset_mel": ([vp, fp, i32, i32, fp, vp], i32),
        "fac_head_begin": ([vp], i32),
        "fac_head_tensor": ([vp, i32, _c.c_char_p, fp, _c.POINTER(_c.c_int64), i32], i32),
        "fac_head_finalize": ([vp, i32, i32, i32, i32, i32], i32),
        "fac_head_forward": ([vp, i32, fp, i32, i32, _c.POINTER(vp), vp], i32),
        "fac_rvq_create": ([vp, i32] + [_c.POINTER(vp)] * 5, i32),
        "fac_rvq_destroy": ([vp, i32], i32),
        "fac_stream_begin": ([vp, i32], i32),
        "fac_stream_encode": ([vp, i32, fp, i32, fp, vp], i32),
        "fac_stream_decode": ([vp, i32, fp, i32, fp, vp], i32),
        "fac_stream_end": ([vp, i32], i32),
        "fac_spectral_loss": ([vp, fp, fp, i32, i32, i32, i32, _c.POINTER(_c.c_int), _c.POINTER(_c.c_int), fp, fp,
                               _c.c_float, _c.c_float, _c.c_float, _c.c_float, fp, vp], i32),
        "fac_l1_loss": ([vp, fp, fp, _c.c_longlong, fp, vp], i32),
        "fac_add3": ([vp, fp, fp, fp, _c.c_longlong, fp, vp], i32),
        "fac_reconstruction_loss": ([vp, fp, fp, i32, i32, fp, fp, vp], i32),
        "fac_rvq_forward": ([vp, i32, fp, i32, i32, i32, fp, i64p, fp, vp], i32),
        "fac_alias_free_act": ([vp, fp, i32, i32, i32, i32, fp, fp, fp, vp], i32),
        "fac_debug_conv": ([vp, fp, fp, fp] + [i32] * 10 + [fp, fp, i32, fp, fp, i32, vp], i32),
        "fac_debug_conv_tc": ([vp, fp, fp, fp] + [i32] * 10 + [fp, fp, i32, fp, fp, i32, i32, vp], i32),
        "fac_debug_resunit": ([vp, fp, fp, fp, fp, fp, fp, fp, i32, i32, i32, i32, i32, fp, vp], i32),
        "fac_debug_tc_phase_clocks": ([vp, _c.POINTER(_c.c_longlong)], i32),
        "fac_debug_tc_producer_clocks": ([vp, _c.POINTER(_c.c_longlong)], i32),
        "fac_debug_tc_trace": ([vp, _c.POINTER(_c.c_longlong)], i32),
        "fac_debug_lstm_pack": ([fp, i32, i32, fp, _c.c_longlong, _c.POINTER(_c.c_int)], _c.c_longlong),
        "fac_debug_convtr_pack": ([fp, i32, i32, i32, i32, fp, _c.c_longlong], _c.c_longlong),
        "fac_debug_pad_map": ([i32, i32, i32, i32, _c.POINTER(_c.c_int), i32], i32),
        "fac_debug_tc_plan": ([i32] * 8 + [_c.POINTER(_c.c_int)], i32),
        "fac_debug_tc_pack": ([fp, i32, i32, i32, i32, i32, fp, _c.c_longlong], _c.c_longlong),
        "fac_debug_lstm_phase_clocks": ([vp, _c.POINTER(_c.c_longlong)], i32),
        "fac_set_option": ([vp, _c.c_char_p, i32], i32),
        "fac_debug_slstm": ([vp, fp, _c.POINTER(vp), i32, i32, i32, fp, vp], i32),
        "fac_debug_tap": ([vp, _c.c_char_p, fp, _c.c_size_t], i32),
        "fac_profile_enable": ([vp, i32], i32),
        "fac_profile_reset": ([vp], i32),
        "fac_profile_get": ([vp, _c.c_char_p, _c.POINTER(_c.c_double), _c.POINTER(_c.c_double),
                             _c.POINTER(_c.c_double), _c.POINTER(_c.c_longlong)], i32),
        "fac_profile_dump": ([vp, _c.c_char_p, _c.c_size_t], _c.c_size_t),
        "fac_workspace_bytes": ([vp], _c.c_size_t),
        "fac_last_launch_count": ([vp], i32),
    }
    for name, (args, res) in sigs.items():
        fn = getattr(L, name)   # AttributeError if the header and the library disagree
        fn.argtypes = args
        fn.restype = res
    _LIB = L
    return L


EXPORTED = ["fac_abi_version", "fac_create", "fac_destroy", "fac_last_error", "fac_load_tensor", "fac_finalize",
            "fac_encode", "fac_encode_frames", "fac_quantize", "fac_decode", "fac_codec_forward",
            "fac_codec_forward_host", "fac_redecode", "fac_redecoder_decode", "fac_voice_convert", "fac_dequantize", "fac_decode_codes", "fac_dataset_mel", "fac_reconstruction_loss", "fac_spectral_loss", "fac_l1_loss", "fac_head_begin", "fac_head_tensor", "fac_head_finalize", "fac_head_forward", "fac_add3", "fac_stream_begin", "fac_stream_encode", "fac_stream_decode", "fac_stream_end", "fac_rvq_create", "fac_rvq_destroy", "fac_rvq_forward", "fac_alias_free_act",
            "fac_debug_conv", "fac_debug_conv_tc", "fac_debug_resunit", "fac_debug_tc_phase_clocks", "fac_debug_tc_producer_clocks", "fac_debug_tc_trace", "fac_debug_lstm_pack", "fac_debug_convtr_pack", "fac_debug_pad_map", "fac_debug_tc_plan", "fac_debug_tc_pack", "fac_debug_lstm_phase_clocks", "fac_set_option", "fac_debug_slstm", "fac_debug_tap", "fac_profile_enable", "fac_profile_reset", "fac_profile_get", "fac_profile_dump",
            "fac_workspace_bytes", "fac_last_launch_count"]


def check(handle, rc, what):
    if rc < 0:
        msg = load().fac_last_error(handle)
        raise FacError(f"{what} failed (status {rc}): {msg.decode() if msg else ''}")
    return rc
