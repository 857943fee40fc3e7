"""ctypes binding of the C ABI declared in include/funcodec_b200.h (the only way Python reaches the kernels).

This is the stub a FunCodec maintainer would add next to funcodec/models/codec_basic.py (INTEGRATION.md).
There is NO fallback: if the shared library is missing or the CUDA call fails, an exception is raised.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int32, c_int64, c_void_p, POINTER, Structure

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfuncodec_b200.so")

FCB_MAX_RATIOS = 8
FCB_NUM_PHASES = 5
PHASE_NAMES = ("encoder_conv", "encoder_lstm", "rvq", "decoder_lstm", "decoder_conv")


class FcbConfig(Structure):
    _fields_ = [("n_ratios", c_int32), ("ratios", c_int32 * FCB_MAX_RATIOS), ("n_filters", c_int32),
                ("dimension", c_int32), ("kernel_size", c_int32), ("last_kernel_size", c_int32),
                ("residual_kernel_size", c_int32), ("lstm_layers", c_int32), ("codebook_size", c_int32),
                ("num_quantizers", c_int32), ("sample_rate", c_int32), ("audio_normalize", c_int32),
                ("gn_eps", c_float), ("arch", c_int32), ("ratios_f", c_int32 * FCB_MAX_RATIOS), ("n_fft", c_int32),
                ("stft_hop", c_int32), ("conv_group_ratio", c_int32), ("tr_conv_group_ratio", c_int32),
                ("n_residual_layers", c_int32), ("dilation_base", c_int32),
                ("norm", c_int32), ("causal", c_int32), ("channels", c_int32)]


FCB_MAX_TAIL_SEGMENTS = 16


class FcbSegmentPlan(Structure):
    _fields_ = [("n_seg", c_int32), ("n_full", c_int32), ("n_tail", c_int32), ("frames_full", c_int32),
                ("decoded_full", c_int32), ("tail_len", c_int32 * FCB_MAX_TAIL_SEGMENTS),
                ("tail_frames", c_int32 * FCB_MAX_TAIL_SEGMENTS), ("total_frames", c_int64)]


class FcbError(RuntimeError):
    pass


# name -> (restype, argtypes); every symbol include/funcodec_b200.h declares
SYMBOLS = {
    "fcb_version": (c_char_p, []),
    "fcb_create": (c_int32, [POINTER(FcbConfig), POINTER(c_void_p)]),
    "fcb_set_tensor": (c_int32, [c_void_p, c_char_p, c_void_p, c_int32, POINTER(c_int64)]),
    "fcb_finalize": (c_int32, [c_void_p]),
    "fcb_num_frames": (c_int32, [c_void_p, c_int32]),
    "fcb_decoded_length": (c_int32, [c_void_p, c_int32]),
    "fcb_num_quantizers_for_bandwidth": (c_int32, [c_void_p, c_double]),
    "fcb_encode": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                             c_void_p, c_void_p]),
    "fcb_decode_emb": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "fcb_decode_codes": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "fcb_roundtrip": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p]),
    "fcb_roundtrip_host": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "fcb_check_errors": (c_int32, [c_void_p, c_void_p]),
    "fcb_launch_count": (c_int64, [c_void_p]),
    "fcb_set_profiling": (c_int32, [c_void_p, c_int32]),
    "fcb_get_phase_ms": (c_int32, [c_void_p, POINTER(c_float)]),
    "fcb_set_option": (c_int32, [c_void_p, c_char_p, c_int32]),
    "fcb_debug_conv1d": (c_int32, [c_void_p, c_char_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p,
                                   POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "fcb_plan_segments": (c_int32, [c_void_p, c_int32, c_int32, c_int32, c_void_p]),
    "fcb_plan_segments_for_hop": (c_int32, [c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "fcb_roundtrip_segmented": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p]),
    "fcb_debug_conv2d": (c_int32, [c_void_p, c_char_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_int64, c_void_p,
                                   POINTER(c_int32), c_void_p]),
    "fcb_last_error": (c_char_p, [c_void_p]),
    "fcb_destroy": (None, [c_void_p]),
}

_lib = None


def load_library(path: str = None) -> ctypes.CDLL:
    """dlopen the in-tree library and bind every declared symbol; raises FcbError when it is absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise FcbError(f"{p} not found: build it with `python -m funcodec_b200.build` (no CPU fallback exists)")
    lib = ctypes.CDLL(p)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)       # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


def check(lib, handle, rc: int, what: str):
    if rc < 0:
        msg = lib.fcb_last_error(handle)
        raise FcbError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")
    return rc
