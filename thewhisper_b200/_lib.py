"""ctypes binding of the C-ABI declared in include/thewhisper_b200.h.

The shared library is built in-tree by `thewhisper_b200.build` (nvcc, sm_100a).  There is no CPU fallback: if the
library is missing or no CUDA device is present, every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_C", "libthewhisper_b200.so")


class BwError(RuntimeError):
    pass


class bw_config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "d_model", "n_heads", "ffn", "enc_layers", "dec_layers", "n_mels", "vocab", "max_source_positions",
        "max_target_positions", "max_audios", "max_beams", "n_align_heads", "max_align_steps", "dtype")]


class bw_decode_opts(C.Structure):
    _fields_ = [
        ("begin_index", C.c_int32), ("eos_token", C.c_int32), ("pad_token", C.c_int32),
        ("timestamp_rules", C.c_int32), ("timestamp_begin", C.c_int32), ("no_timestamps_token", C.c_int32),
        ("max_initial_timestamp_index", C.c_int32),
        ("suppress_tokens", C.POINTER(C.c_int32)), ("n_suppress", C.c_int32),
        ("begin_suppress_tokens", C.POINTER(C.c_int32)), ("n_begin_suppress", C.c_int32),
        ("record_alignment", C.c_int32),
    ]


# every symbol include/thewhisper_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I = C.c_int32
_F = C.c_float
SYMBOLS = {
    "bw_last_error": (C.c_char_p, []),
    "bw_abi_version": (C.c_int, []),
    "bw_device_count": (C.c_int, []),
    "bw_runtime_flags": (C.c_int, []),
    "bw_engine_create": (C.c_int, [C.POINTER(bw_config), C.POINTER(_P)]),
    "bw_engine_destroy": (None, [_P]),
    "bw_engine_set_tensor": (C.c_int, [_P, C.c_char_p, _P]),
    "bw_engine_set_mel_filters": (C.c_int, [_P, _P]),
    "bw_engine_set_alignment_heads": (C.c_int, [_P, _P, _I]),
    "bw_engine_finalize": (C.c_int, [_P]),
    "bw_engine_buffer": (C.c_int, [_P, C.c_char_p, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    "bw_logmel": (C.c_int, [_P, _P, _I, _I, _P, _P]),
    "bw_set_mel": (C.c_int, [_P, _P, _I, _P]),
    "bw_encode": (C.c_int, [_P, _I, _P]),
    "bw_decode_begin": (C.c_int, [_P, _I, _I, _P, _I, C.POINTER(bw_decode_opts), _P]),
    "bw_decode_run": (C.c_int, [_P, _I, _P]),
    "bw_decode_kernel_launches": (C.c_longlong, [_P]),
    "bw_decode_read": (C.c_int, [_P, _P, _P, _P, _P]),
    "bw_decode_reorder": (C.c_int, [_P, _P, _P, _P]),
    "bw_decode_beam_step": (C.c_int, [_P, _P, _P, _P, _P]),
    "bw_word_timestamps": (C.c_int, [_P, _I, _I, _I, C.c_double, _P, _P]),
    "bw_word_timestamps_batch": (C.c_int, [_P, _I, _P, _P, _P, C.c_double, _P, _I, _P]),
    "bw_word_timestamps_gather": (C.c_int, [_P, _I, _P, _I, _P, _P, C.c_double, _P, _I, _P]),
    "bw_host_merge_overlapping": (C.c_int, [_P, _P, _I, _P, _P, _P, _P]),
    "bw_host_vocab_create": (C.c_int, [_P, _P, _I, _P, C.c_char_p, _I, _I, _I, _I, _I, _I, _I, _P]),
    "bw_host_vocab_destroy": (None, [_P]),
    "bw_host_decode_asr": (C.c_int, [_P, _P, _P, _I, _P, _P, _P, _P, _I, _I, C.c_double, _I, _P, _P]),
    "bw_op_gemm": (C.c_int, [_P, _P, _I, _I, _I, _P, _F, _I, _P, _P, _I, _I, _I, _P]),
    "bw_op_gemm_splitk": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _P, C.POINTER(_I), _P]),
    "bw_op_gemm_dec": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P, C.POINTER(_I), _P]),
    "bw_op_gelu_bias": (C.c_int, [_P, _I, _P, _P, _I, _I, _P]),
    "bw_op_resid_ln": (C.c_int, [_P, _P, _I, _P, _P, _P, _P, _I, _I, _P]),
    "bw_op_attn_enc": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "bw_op_layernorm": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "bw_op_gemv": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P, _F, _I, _P, _P, _P]),
    "bw_op_self_attn": (C.c_int, [_P, _I, _P, _F, _P, _P, _P, _I, _P, _I, _P, _I, _I, _I, _I, _P]),
    "bw_op_cross_attn": (C.c_int, [_P, _I, _P, _F, _P, _P, _P, _I, _P, _P, _P, _I, _I, _I, _I, _P, _P, _I, _I, _I, _P, _I, _I, _P]),
}

_lib: Optional[C.CDLL] = None


def load(build_if_missing: bool = False) -> C.CDLL:
    """Load the library and bind every declared symbol; raises BwError when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if build_if_missing:
            from . import build as _build

            _build.build()
        else:
            raise BwError(f"{LIB_PATH} not found: run `python -m thewhisper_b200.build` (nvcc, sm_100a). "
                          "thewhisper_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    if lib.bw_abi_version() != 2:
        raise BwError("ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().bw_last_error()
        raise BwError((msg or b"unknown error").decode("utf-8", "replace") + f" (code {rc})")


_cudart = None


def device_copy(dst_ptr: int, src_ptr: int, nbytes: int) -> None:
    """cudaMemcpy(device -> device) through the CUDA runtime already loaded in the process."""
    global _cudart
    if _cudart is None:
        _cudart = C.CDLL("libcudart.so.12")
        _cudart.cudaMemcpy.restype = C.c_int
        _cudart.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    rc = _cudart.cudaMemcpy(C.c_void_p(dst_ptr), C.c_void_p(src_ptr), nbytes, 3)
    if rc != 0:
        raise BwError(f"cudaMemcpy failed with code {rc}")
