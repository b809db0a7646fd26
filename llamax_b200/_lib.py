"""ctypes binding of the C-ABI library declared in include/llamax_b200.h.

The library is the product path: there is no PyTorch/CPU fallback. If it is missing, importing an op fails
loudly with the build command.
"""

import ctypes
import os
import threading
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# LLAMAX_B200_LIB: load another build of the same library (tools/attn_trace.py uses an instrumented one)
LIB_PATH = os.environ.get("LLAMAX_B200_LIB") or os.path.join(_HERE, "csrc", "libllamax_b200.so")

P = c_void_p
I64 = c_int64
I32 = c_int32


class Epilogue(Structure):
    """llamax_epilogue_t"""

    _fields_ = [
        ("lora_h", P),
        ("ldh", I64),
        ("lora_b", P),
        ("lora_rank", I32),
        ("lora_scale", c_float),
        ("resid", P),
        ("ldr", I64),
        ("seg_n0", I32),
        ("seg_n1", I32),
        ("rope", P),
        ("rope_S", I32),
        ("rope_cols", I32),
    ]


EP = POINTER(Epilogue)

MAX_COPY_JOBS = 64
LORA_WGRAD_MAX_SPLITS = 32


class CopyJob(Structure):
    """llamax_copy_job_t"""

    _fields_ = [
        ("src", P),
        ("dst", P),
        ("src_ld", I64),
        ("dst_ld", I64),
        ("rows", I32),
        ("cols", I32),
        ("scale", c_float),
        ("flags", I32),
    ]

# name -> argtypes (every function returns int except llamax_last_error)
SIGNATURES = {
    "llamax_version": [],
    "llamax_set_device": [c_int],
    "llamax_set_gemm_cta_group": [c_int],
    "llamax_int8_gemm_dequant": [P, I64, P, I64, P, P, P, I64, I64, I64, I64, EP, P],
    "llamax_int8_gemm_s32": [P, I64, P, I64, P, I64, I64, I64, I64, P],
    "llamax_bf16_gemm": [P, I64, P, I64, P, I64, I64, I64, I64, P, c_int, EP, P],
    "llamax_bf16_gemm_swiglu_bwd": [P, I64, P, I64, I64, I64, I64, EP, P, I64, P, I64, P, P],
    "llamax_bf16_gemm_tn": [P, I64, P, I64, P, I64, I64, I64, I64, P],
    "llamax_bf16_gemm_rowdot": [P, I64, P, I64, P, I64, I64, I64, I64, EP, P, I64, P, I64, P],
    "llamax_bf16_int8_gemm": [P, I64, P, I64, P, c_int, P, I64, P, I64, I64, I64, I64, I64, EP, P],
    "llamax_bf16_int8_gemm_swiglu_bwd": [P, I64, P, I64, P, I64, I64, I64, EP, P, I64, P, I64, P, P],
    "llamax_dequant_weight": [P, P, P, I64, I64, I64, c_int, c_int, P],
    "llamax_rowquant_int8": [P, I64, P, P, I64, I64, P],
    "llamax_rowquant_int8_colscale": [P, I64, P, P, P, I64, I64, P],
    "llamax_rmsnorm_fwd": [P, P, P, P, P, P, I64, I64, c_float, P],
    "llamax_rmsnorm_bwd": [P, P, P, P, P, P, P, I32, I64, I64, P],
    "llamax_reduce_partials": [P, P, I32, I64, P],
    "llamax_swiglu_fwd": [P, P, I64, P, P, P, I64, I64, P],
    "llamax_swiglu_bwd": [P, P, P, I64, P, P, I64, P, I64, I64, P],
    "llamax_rope_inplace": [P, I64, P, I64, I64, I32, I32, c_int, P],
    "llamax_attn_fwd": [P, I64, P, I64, P, I64, P, I64, P, I64, I64, I32, I32, I32, I64, P, P, c_float, P],
    "llamax_attn_bwd": [P, I64, P, I64, P, I64, P, I64, P, P, I64, P, I64, P, I64, P, I64, P, P,
                        I64, I64, I32, I32, I32, I64, P, P, P, c_float, P, P],
    "llamax_attn_bwd_deterministic": [P, I64, P, I64, P, I64, P, I64, P, P, I64, P, I64, P, I64, P, I64, P,
                                      I64, I64, I32, I32, I32, I64, P, P, P, c_float, P, P],
    "llamax_lora_wgrad": [P, I64, P, I64, P, I64, I64, I32, c_float, P],
    "llamax_lora_wgrad_deterministic": [P, I64, P, I64, P, P, I64, I64, I32, c_float, P],
    "llamax_lora_bwd_pair": [P, I64, P, I64, P, I64, P, I64, P, I64, P, P, I64, I64, I32, c_float, P],
    "llamax_gelu_bias_fwd": [P, P, P, I64, I64, I32, I32, I32, P],
    "llamax_gelu_bwd": [P, P, P, I64, I64, I32, I32, I32, P],
    "llamax_conv_s2k3_col2im": [P, P, I64, I64, I64, P],
    "llamax_batched_copy": [POINTER(CopyJob), I32, P],
    "llamax_cross_entropy": [P, I64, P, P, P, I64, I64, c_int, P],
    "llamax_cross_entropy_rows": [P, I64, P, P, P, I64, I64, c_int, P],
}

_lib = None
_lock = threading.Lock()


class LlamaxError(RuntimeError):
    pass


def load():
    """Load libllamax_b200.so (once). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise LlamaxError(
                f"{LIB_PATH} not found: the CUDA extension is the only implementation of this path "
                "(no fallback). Build it with `python -m llamax_b200.build`."
            )
        lib = ctypes.CDLL(LIB_PATH)
        lib.llamax_last_error.restype = c_char_p
        lib.llamax_last_error.argtypes = []
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is missing
            fn.restype = c_int
            fn.argtypes = argtypes
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().llamax_last_error().decode("utf-8", "replace")
        raise LlamaxError(f"{what} failed (code {rc}): {msg}")
