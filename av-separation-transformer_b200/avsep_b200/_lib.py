"""ctypes binding of libavsep.so (C ABI declared in include/avsep.h).

There is no CPU fallback: if the CUDA library has not been built, importing the engine fails loudly.
Build it with ``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C av-separation-transformer_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libavsep.so")

PREC_BF16, PREC_TF32 = 0, 1
DTYPE_F32, DTYPE_I64 = 0, 1


class AvsepConfig(C.Structure):
    _fields_ = [
        ("freq_bins", C.c_int32), ("d_model", C.c_int32), ("nhead", C.c_int32),
        ("num_encoder_layers", C.c_int32), ("num_fusion_layers", C.c_int32), ("num_speakers", C.c_int32),
        ("precision", C.c_int32), ("device", C.c_int32),
    ]


class AvsepSynthConfig(C.Structure):
    _fields_ = [
        ("num_samples_audio", C.c_int32), ("duration", C.c_double), ("n_fft", C.c_int32), ("hop_length", C.c_int32),
        ("num_frames", C.c_int32), ("frame_h", C.c_int32), ("frame_w", C.c_int32), ("num_speakers", C.c_int32),
    ]


_P = C.c_void_p
_I = C.c_int32

# name -> (restype, argtypes); must list every symbol include/avsep.h declares
SIGNATURES = {
    "avsep_create": (C.c_int, [C.POINTER(AvsepConfig), C.POINTER(_P)]),
    "avsep_destroy": (None, [_P]),
    "avsep_last_error": (C.c_char_p, [_P]),
    "avsep_set_weight": (C.c_int, [_P, C.c_char_p, _P, _I, C.POINTER(C.c_int64), _I]),
    "avsep_finalize_weights": (C.c_int, [_P, _P]),
    "avsep_workspace_bytes": (C.c_size_t, [_P, _I, _I, _I, _I, _I]),
    "avsep_forward": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, C.c_size_t, _P]),
    "avsep_forward_varlen": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, C.c_size_t, _P]),
    "avsep_forward_host": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "avsep_forward_host_async": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P]),
    "avsep_host_wait": (C.c_int, [_P, _I]),
    "avsep_last_launch_count": (C.c_int64, [_P]),
    "avsep_audio_encoder": (C.c_int, [_P, _P, _I, _I, _P, _P]),
    "avsep_visual_encoder": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "avsep_fusion": (C.c_int, [_P, _P, _P, _I, _I, _I, _P, _P]),
    "avsep_decoder": (C.c_int, [_P, _P, _P, _I, _I, _P, _P, _P]),
    "avsep_set_debug": (C.c_int, [_P, _I]),
    "avsep_debug_get_stage": (C.c_int, [_P, C.c_char_p, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "avsep_set_profile": (C.c_int, [_P, _I]),
    "avsep_profile_report": (C.c_int, [_P, C.c_char_p, C.c_size_t, _I]),
    "avsep_test_gemm": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "avsep_test_gemm_ln": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "avsep_set_option": (C.c_int, [_P, C.c_char_p, _I]),
    "avsep_test_gemm_trace": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "avsep_test_ffn_fused": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _I, _P]),
    "avsep_test_ffn_fused_trace": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _I, _P, _P]),
    "avsep_test_conv1d": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _P]),
    "avsep_test_attention": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "avsep_test_add_layernorm": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _P]),
    "avsep_test_visual_cnn": (C.c_int, [_P, _P, _I, _I, _I, _P, _P]),
    "avsep_test_visual_cnn_trace": (C.c_int, [_P, _P, _I, _P, _P, _P]),
    "avsep_synth_batch": (C.c_int, [_P, C.POINTER(AvsepSynthConfig), _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "avsep_eval_snr": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "avsep_stft": (C.c_int, [_P, _P, _I, _I, _I, _I, _P, _P, _P]),
    "avsep_istft": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "avsep_stft_varlen": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "avsep_istft_varlen": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P]),
    "avsep_test_xformer_stack": (C.c_int, [_P, _I, _P, _P, _I, _I, _P, _P, _I, _P, _P]),
    "avsep_test_fusion_decoder": (C.c_int, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _P]),
    "avsep_shared_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P), C.c_char_p]),
    "avsep_shared_free": (C.c_int, [_P, _P]),
    "avsep_shared_open": (C.c_int, [_P, C.c_char_p, C.POINTER(_P)]),
    "avsep_shared_close": (C.c_int, [_P, _P]),
    "avsep_copy_async": (C.c_int, [_P, _P, _P, C.c_size_t, _P]),
    "avsep_separate": (C.c_int, [_P, _P, _P, _I, _I, _P, _P]),
    "avsep_flag_signal": (C.c_int, [_P, C.POINTER(_P), _I, C.c_uint32, _P]),
    "avsep_flag_wait": (C.c_int, [_P, C.POINTER(_P), _I, C.c_uint32, C.c_double, _P]),
}
IPC_HANDLE_BYTES = 64

_lib = None


def load():
    """Load libavsep.so once and attach the prototypes. Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built and there is no CPU fallback. "
            "Run `make -C av-separation-transformer_b200/csrc` (needs nvcc, targets sm_100a).")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here = header and library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
