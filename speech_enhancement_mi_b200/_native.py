"""ctypes binding of libse_b200.so (C-ABI declared in include/se_b200.h).

There is no CPU fallback: if the library is missing, cannot be loaded, or no B200 is present, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libse_b200.so")
SE_MAX_LEVELS = 8

SE_VARIANT_CRN_ELU = 0
SE_VARIANT_DISTILLED = 1
SE_PRECISION_FP32 = 0
SE_PRECISION_TF32 = 1
SE_PRECISION_FP16 = 2
SE_PRECISION_3XTF32 = 3


class SeCrnConfig(C.Structure):
    _fields_ = [
        ("num_inputs", C.c_int32),
        ("num_freqs", C.c_int32),
        ("num_levels", C.c_int32),
        ("num_channels", C.c_int32 * SE_MAX_LEVELS),
        ("hidden", C.c_int32),
        ("num_layers", C.c_int32),
        ("kernel_size", C.c_int32),
        ("segment_length", C.c_int32),
        ("n_fft", C.c_int32),
        ("win_length", C.c_int32),
        ("hop_length", C.c_int32),
        ("variant", C.c_int32),
        ("precision", C.c_int32),
        ("max_streams", C.c_int32),
        ("training", C.c_int32),
    ]


class SeFsnConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("num_freqs", "num_mics", "fb_hidden", "sb_hidden", "num_layers",
                                         "sb_num_neighbors", "fb_num_neighbors", "max_streams", "precision")]


_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_PI = C.POINTER(C.c_int)
_PI32 = C.POINTER(C.c_int32)

# name -> (restype, argtypes); must list every symbol of include/se_b200.h (tests/test_abi.py checks this)
SIGNATURES = {
    "se_ctx_create": (_I, [C.POINTER(_P), _I, C.POINTER(SeCrnConfig)]),
    "se_ctx_destroy": (_I, [_P]),
    "se_last_error": (C.c_char_p, []),
    "se_version": (C.c_char_p, []),
    "se_crn_num_params": (_I, [_P]),
    "se_crn_param_name": (C.c_char_p, [_P, _I]),
    "se_crn_param_numel": (_L, [_P, _I]),
    "se_crn_bind_weights": (_I, [_P, C.POINTER(_P), _I, _P]),
    "se_crn_state_reset": (_I, [_P, _I, _I, _P]),
    "se_crn_state_bytes_per_stream": (_L, [_P]),
    "se_crn_state_layout": (C.c_uint64, [_P]),
    "se_crn_state_export": (_I, [_P, _PI32, _I, _P, _P]),
    "se_crn_state_import": (_I, [_P, _PI32, _I, _P, C.c_uint64, _P]),
    "se_crn_process_chunk": (_I, [_P, _P, _L, _L, _P, _L, _I, _P]),
    "se_crn_realtime_process": (_I, [_P, _P, _I, _L, _I, _P, _P]),
    "se_crn_realtime_process_host": (_I, [_P, _P, _I, _L, _I, _P]),
    "se_stft_trans": (_I, [_P, _P, _I, _P, _P]),
    "se_istft_trans": (_I, [_P, _P, _I, _P, _P]),
    "se_crn_forward_chunk": (_I, [_P, _P, _P, _I, _P]),
    "se_segmentation": (_I, [_P, _I, _I, _L, _I, _P, _PI, _PI, _P]),
    "se_chunk_grid": (_I, [_L, _I, _PI, _PI]),
    "se_over_add": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "se_crn_launches_per_chunk": (_I, [_P]),
    "se_crn_set_graph": (_I, [_P, _I]),
    "se_crn_time_stage": (_I, [_P, C.c_char_p, _I, _I, C.POINTER(C.c_float)]),
    "se_fsn_create": (_I, [C.POINTER(_P), _I, C.POINTER(SeFsnConfig)]),
    "se_fsn_destroy": (_I, [_P]),
    "se_fsn_num_params": (_I, [_P]),
    "se_fsn_param_name": (C.c_char_p, [_P, _I]),
    "se_fsn_param_numel": (_L, [_P, _I]),
    "se_fsn_bind_weights": (_I, [_P, C.POINTER(_P), _I, _P]),
    "se_fsn_reset_state": (_I, [_P, _I, _I, _P]),
    "se_fsn_state_bytes_per_stream": (_L, [_P]),
    "se_fsn_state_layout": (C.c_uint64, [_P]),
    "se_fsn_state_export": (_I, [_P, _PI32, _I, _P, _P]),
    "se_fsn_state_import": (_I, [_P, _PI32, _I, _P, C.c_uint64, _P]),
    "se_fsn_forward_chunk": (_I, [_P, _P, _P, _I, _P]),
    "se_fsn_process_chunk": (_I, [_P, _P, _L, _L, _P, _L, _I, _P]),
    "se_fsn_apply_mask": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "se_fsn_planes": (_I, [_P, _I, _I, _I, _I, _P, _P, _P]),
    "se_fsn_realtime_process": (_I, [_P, _P, _P, _I, _L, _I, _I, _P, _P, _P, _P, _P]),
    "se_unfold": (_I, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "se_cal_si_snr": (_I, [_P, _P, _P, _I, _L, _P, _P]),
    "se_stoi_loss": (_I, [_P, _P, _P, _I, _L, _P, _P]),
    "se_crn_num_kernels": (_I, [_P]),
    "se_crn_kernel_info": (_I, [_P, _I, C.c_char_p, _I, C.POINTER(C.c_double), C.POINTER(C.c_double), _PI]),
    "se_crn_time_kernel": (_I, [_P, _I, _I, _I, C.POINTER(C.c_float)]),
    "se_crn_num_theta": (_L, [_P]),
    "se_crn_param_offset": (_L, [_P, _I]),
    "se_crn_bind_weights_flat": (_I, [_P, _P, _P]),
    "se_crn_train_forward": (_I, [_P, _P, _I, _L, _I, _P, _P]),
    "se_crn_train_backward": (_I, [_P, _P, _P, _P]),
    "se_crn_train_num_taps": (_I, [_P]),
    "se_crn_train_tap_shape": (_I, [_P, _I, _P, _P, _P]),
    "se_crn_train_tap": (_I, [_P, _I, _P, _P]),
    "se_crn_train_backward_taps": (_I, [_P, _P, _P, _I, _P, _P]),
    "se_crn_train_backward_input": (_I, [_P, _P, _P, _P, _I, _P, _P, _P]),
    "se_loss_terms_grad": (_I, [_P, _P, _P, _I, _L, _P, _P, _P, _P]),
    "se_axpby_dev": (_I, [_P, _P, _P, _P, _P, _L, _P]),
    "se_clip_adam_step": (_I, [_P, _P, _P, _P, _L, C.c_float, C.c_float, C.c_float, C.c_float, _I, C.c_float,
                               C.c_float, _P, _P]),
    "se_debug_read": (_I, [_P, C.c_char_p, _I, _P, _L, C.POINTER(C.c_int)]),
    "se_debug_mask_spectrum": (_I, [_P, _P, _P, _P, _I]),
    "se_debug_gemm_counters": (_I, [C.POINTER(C.c_uint64), _I]),
    "se_debug_gru_counters": (_I, [C.POINTER(C.c_uint64), _I]),
}

_lib = None


def lib():
    """Load the shared library (once).  Raises if it has not been built -- never falls back to anything."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m speech_enhancement_mi_b200.build` "
                "(there is no CPU / PyTorch fallback for this path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().se_last_error()
        raise RuntimeError(f"{what} failed (status {rc}): {msg.decode() if msg else '?'}")


def chunk_grid(length: int, K: int):
    """(gap, n_chunks) of utility.segmentation for a signal of `length` samples (reference utility.py:325-327,357-368)."""
    gap, n = C.c_int(0), C.c_int(0)
    check(lib().se_chunk_grid(length, K, C.byref(gap), C.byref(n)), "se_chunk_grid")
    return gap.value, n.value
