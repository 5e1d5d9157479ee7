"""ctypes binding of libf5tts_b200.so (C ABI declared in include/f5tts_b200.h).

There is NO fallback: if the shared library is missing or the device is not sm_100 the import of any
operator raises.  Build with ``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C f5_tts_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("F5_LIB") or os.path.join(_HERE, "libf5tts_b200.so")  # F5_LIB: diagnostic (trace) build

c_void_p, c_int, c_float, c_size_t, c_ll = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_longlong

ACT_NONE, ACT_GELU_TANH, ACT_GELU_ERF, ACT_MISH = 0, 1, 2, 3
EPI_F16, EPI_F32, EPI_RESID, EPI_QKV_ROPE = 0, 1, 2, 3
ODE_EULER, ODE_MIDPOINT = 0, 1
ODE_METHODS = {"euler": ODE_EULER, "midpoint": ODE_MIDPOINT}


class GemmArgs(C.Structure):
    _fields_ = [
        ("rows", c_int), ("batches", c_int), ("n_out", c_int), ("k", c_int), ("lda", c_int), ("ldw", c_int),
        ("bn", c_int), ("epi", c_int), ("act", c_int), ("conv_taps", c_int), ("cta_pair", c_int),
        ("bias", c_void_p), ("out", c_void_p), ("out16b", c_void_p), ("resid", c_void_p), ("ldo", c_int),
        ("gate", c_void_p), ("step_ptr", c_void_p), ("gate_step_stride", c_ll), ("row_len", c_void_p),
        ("seq", c_int), ("rope_cos", c_void_p), ("rope_sin", c_void_p), ("inner", c_int), ("pe_heads", c_int),
        ("weights_static", c_int),
        ("skip_padded_tiles", c_int),
    ]


class VocosWeights(C.Structure):
    _fields_ = [
        ("embed_w", c_void_p), ("embed_b", c_void_p), ("norm_w", c_void_p), ("norm_b", c_void_p),
        ("dw_w", c_void_p * 8), ("dw_b", c_void_p * 8), ("ln_w", c_void_p * 8), ("ln_b", c_void_p * 8),
        ("pw1_w", c_void_p * 8), ("pw1_b", c_void_p * 8), ("pw2_w", c_void_p * 8), ("pw2_b", c_void_p * 8),
        ("gamma", c_void_p * 8), ("final_w", c_void_p), ("final_b", c_void_p), ("head_w", c_void_p),
        ("head_b", c_void_p), ("dim", c_int), ("inter", c_int), ("layers", c_int), ("n_mels", c_int),
    ]


class Arch(C.Structure):
    _fields_ = [(n, c_int) for n in ("backbone", "dim", "depth", "heads", "dim_head", "ff_inner", "mel_dim", "text_dim",
                                     "text_num_embeds", "conv_layers", "text_mask_padding", "pe_attn_head",
                                     "attn_mask_enabled")]


class LayerWeights(C.Structure):
    _fields_ = [(n, c_void_p) for n in ("w_qkv", "b_qkv", "w_out", "b_out", "w_ff1", "b_ff1", "w_ff2", "b_ff2",
                                        "w_skip", "g_attn", "g_ff")]


class TextBlock(C.Structure):
    _fields_ = [(n, c_void_p) for n in ("dw_w", "dw_b", "ln_w", "ln_b", "pw1_w", "pw1_b", "grn_gamma", "grn_beta",
                                        "pw2_w", "pw2_b")]


class Weights(C.Structure):
    _fields_ = [
        ("time_w0", c_void_p), ("time_b0", c_void_p), ("time_w1", c_void_p), ("time_b1", c_void_p),
        ("text_table", c_void_p), ("text_blocks", TextBlock * 8),
        ("proj_w", c_void_p), ("proj_b", c_void_p), ("proj_kpad", c_int),
        ("conv_w", c_void_p * 2), ("conv_b", c_void_p * 2),
        ("mod_w", c_void_p), ("mod_b", c_void_p),
        ("layers", C.POINTER(LayerWeights)), ("g_out", c_void_p), ("out_w", c_void_p), ("out_b", c_void_p),
    ]


class SampleArgs(C.Structure):
    _fields_ = [
        ("B", c_int), ("N", c_int), ("nt", c_int), ("steps", c_int),
        ("text", c_void_p), ("step_cond", c_void_p), ("y", c_void_p), ("duration", c_void_p),
        ("t", C.POINTER(c_float)), ("cfg_strength", c_float), ("trajectory", c_void_p), ("use_graph", c_int),
        ("v_out", c_void_p), ("exact_varlen", c_int), ("ode_method", c_int),
    ]


_lock = threading.Lock()
_lib = None


class F5LibraryError(RuntimeError):
    pass


def lib():
    """Load the shared library once; raise loudly when it (or a Blackwell GPU) is missing."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise F5LibraryError(
                f"{LIB_PATH} not found: the B200 CUDA library is not built (run __graft_entry__.build()). "
                "There is no CPU / PyTorch fallback for this path.")
        L = C.CDLL(LIB_PATH)
        L.f5_version.restype = c_int
        L.f5_last_error.restype = C.c_char_p
        L.f5_launch_count.restype = C.c_ulonglong
        L.f5_gemm.argtypes = [c_void_p, c_void_p, C.POINTER(GemmArgs), c_void_p]
        L.f5_gemm_tile.argtypes = [C.POINTER(GemmArgs), C.POINTER(c_int), C.POINTER(c_int)]
        L.f5_attention.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_float, c_void_p]
        L.f5_row_norm.argtypes = [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]
        L.f5_mel_spectrogram.argtypes = [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p]
        L.f5_vocos_workspace_bytes.argtypes = [c_int, c_int]
        L.f5_vocos_workspace_bytes.restype = c_size_t
        L.f5_vocos_decode.argtypes = [C.POINTER(VocosWeights), c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p,
                                      c_void_p]
        L.f5_engine_create.argtypes = [C.POINTER(Arch), C.POINTER(Weights), C.POINTER(c_void_p)]
        L.f5_engine_destroy.argtypes = [c_void_p]
        L.f5_engine_destroy.restype = None
        L.f5_sample_workspace_bytes.argtypes = [c_void_p, c_int, c_int, c_int, c_float]
        L.f5_sample_workspace_bytes.restype = c_size_t
        L.f5_sample.argtypes = [c_void_p, C.POINTER(SampleArgs), c_void_p, c_size_t, c_void_p]
        L.f5_sample_flops.argtypes = [c_void_p, c_int, c_int, c_int, c_float]
        L.f5_sample_flops.restype = C.c_double
        for name in ("f5_gemm", "f5_gemm_tile", "f5_attention", "f5_row_norm", "f5_mel_spectrogram", "f5_vocos_decode",
                     "f5_engine_create", "f5_sample"):
            getattr(L, name).restype = c_int
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().f5_last_error().decode("utf-8", "replace")
        raise F5LibraryError(f"{what} failed (rc={rc}): {msg}")


def launch_count() -> int:
    return int(lib().f5_launch_count())


EXPORTED_SYMBOLS = [
    "f5_version", "f5_last_error", "f5_launch_count", "f5_debug_gemm_trace", "f5_debug_attn_trace", "f5_gemm", "f5_gemm_tile", "f5_attention", "f5_row_norm", "f5_mel_spectrogram",
    "f5_vocos_workspace_bytes", "f5_vocos_decode", "f5_engine_create", "f5_engine_destroy",
    "f5_sample_workspace_bytes", "f5_sample", "f5_sample_flops",
]
