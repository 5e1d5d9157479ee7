"""Thin torch-tensor wrappers over the kernel-level C entry points (used by parity tests and the vocoder).

Every function raises if the CUDA library is missing or the tensors are not on a CUDA device.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import (ACT_GELU_ERF, ACT_GELU_TANH, ACT_MISH, ACT_NONE, EPI_F16, EPI_F32, EPI_QKV_ROPE,  # noqa: F401
                   EPI_RESID)


def _stream(t: torch.Tensor):
    return torch.cuda.current_stream(t.device).cuda_stream


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.F5LibraryError("B200 operators take CUDA tensors only; there is no CPU fallback")


def _rows(t: torch.Tensor, shape, dtype, what: str) -> int:
    """Row stride of a caller-provided 2-D operand whose rows are contiguous (it may be a column slice)."""
    assert t.shape == shape and t.dtype == dtype and t.stride(1) == 1, (what, t.shape, t.dtype, t.stride())
    return t.stride(0)


def linear(a: torch.Tensor, w: torch.Tensor, bias=None, *, epi=EPI_F16, act=ACT_NONE, bn=0, pair=0, resid=None, gate=None,
           row_len=None, seq=0, rope=None, inner=0, pe_heads=0, out16b=False, static_w=False, out=None,
           skip_padded=False, step_ptr=None, gate_stride=0):
    """C = epilogue(a @ w.T).  a fp16 [M, K], w fp16 [N, K]; each may be row-strided (a column slice of a wider tensor).
    static_w: w is a model weight (not produced by the preceding kernel) -> its tiles may be prefetched early.
    out: caller-allocated output [M, N] (fp16, or fp32 for EPI_F32), row-strided like a; allocated when None.
    out16b (EPI_F32): True allocates the masked fp16 copy, a tensor is used as it (same row stride as out).
    skip_padded: tiles whose rows all lie past row_len of their sample are not computed (needs row_len and seq).
    step_ptr / gate_stride: the RESID gate row is gate + (*step_ptr) * gate_stride (device int32 step counter).
"""
    _need_cuda(a, w, bias, resid, gate, out, step_ptr)
    M, K = a.shape
    N = w.shape[0]
    g = _lib.GemmArgs()
    g.rows, g.batches, g.n_out, g.k, g.bn, g.epi, g.act = M, 1, N, K, bn, epi, act
    g.lda = _rows(a, (M, K), torch.float16, "a")
    g.ldw = _rows(w, (N, K), torch.float16, "w")
    g.cta_pair = pair
    g.bias = _ptr(bias)
    out2 = None
    if epi == EPI_RESID:
        assert resid is not None and out is None
        out = resid
        g.ldo = _rows(resid, (M, N), torch.float32, "resid")
        g.resid = resid.data_ptr()
    else:
        dt = torch.float32 if epi == EPI_F32 else torch.float16
        if out is None:
            out = torch.empty((M, N), dtype=dt, device=a.device)
        g.ldo = _rows(out, (M, N), dt, "out")
        g.out = out.data_ptr()
        if epi == EPI_F32 and out16b is not False:
            out2 = torch.empty((M, N), dtype=torch.float16, device=a.device) if out16b is True else out16b
            assert _rows(out2, (M, N), torch.float16, "out16b") == g.ldo
            g.out16b = out2.data_ptr()
    g.gate = _ptr(gate)
    g.step_ptr = _ptr(step_ptr)
    g.gate_step_stride = gate_stride
    g.row_len = _ptr(row_len)
    g.seq = seq
    g.skip_padded_tiles = 1 if skip_padded else 0
    if rope is not None:
        g.rope_cos, g.rope_sin = rope[0].data_ptr(), rope[1].data_ptr()
    g.inner, g.pe_heads = inner, pe_heads
    g.weights_static = 1 if static_w else 0
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().f5_gemm(a.data_ptr(), w.data_ptr(), C.byref(g), _stream(a)), "f5_gemm")
    return (out, out2) if out2 is not None else out


def gemm_tile(M: int, N: int, K: int, epi=EPI_F16, act=ACT_NONE, bn=0, pair=0):
    """(tile width, cta_pair) the planner runs this GEMM shape with."""
    g = _lib.GemmArgs()
    g.rows, g.batches, g.n_out, g.k, g.bn, g.epi, g.act, g.cta_pair = M, 1, N, K, bn, epi, act, pair
    b, pr = C.c_int(0), C.c_int(0)
    _lib.check(_lib.lib().f5_gemm_tile(C.byref(g), C.byref(b), C.byref(pr)), "f5_gemm_tile")
    return b.value, pr.value


def grouped_conv31(x: torch.Tensor, w_packed: torch.Tensor, bias, *, resid=None, row_len=None, out=None,
                   skip_padded=False):
    """Conv1d(k=31, groups=D/64, pad=15) + bias + (mask) + Mish over x fp16 [B, N, D]; w_packed fp16 [31, D, 64].
    resid given: resid += result (fp32, in place) else returns fp16 [B, N, D] (into `out` when given, contiguous).
    skip_padded: 128-row tiles starting at or past row_len[b] are not computed."""
    _need_cuda(x, w_packed, bias, resid, row_len, out)
    B, N, D = x.shape
    g = _lib.GemmArgs()
    g.rows, g.batches, g.n_out, g.lda, g.conv_taps, g.act = N, B, D, D, 31, ACT_MISH
    g.bias = _ptr(bias)
    g.ldo, g.seq, g.row_len = D, N, _ptr(row_len)
    g.skip_padded_tiles = 1 if skip_padded else 0
    g.weights_static = 1
    if resid is None:
        if out is None:
            out = torch.empty((B, N, D), dtype=torch.float16, device=x.device)
        assert out.shape == (B, N, D) and out.dtype == torch.float16 and out.is_contiguous()
        g.epi, g.out = EPI_F16, out.data_ptr()
    else:
        out = resid
        g.epi, g.resid = EPI_RESID, resid.data_ptr()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().f5_gemm(x.data_ptr(), w_packed.data_ptr(), C.byref(g), _stream(x)), "f5_gemm(conv)")
    return out


def attention(qkv: torch.Tensor, batches: int, seq: int, heads: int, kv_len=None, scale=None, out=None) -> torch.Tensor:
    """qkv fp16 [batches*seq, 3*heads*64] -> fp16 [batches*seq, heads*64] (into `out` when given, contiguous).
    With kv_len, query blocks of 256 rows at or past kv_len[b] are not written."""
    _need_cuda(qkv, kv_len, out)
    assert qkv.dtype == torch.float16 and qkv.is_contiguous() and qkv.shape == (batches * seq, 3 * heads * 64)
    if out is None:
        out = torch.empty((batches * seq, heads * 64), dtype=torch.float16, device=qkv.device)
    assert out.shape == (batches * seq, heads * 64) and out.dtype == torch.float16 and out.is_contiguous()
    scale = 0.125 if scale is None else scale
    with torch.cuda.device(qkv.device):
        _lib.check(_lib.lib().f5_attention(qkv.data_ptr(), out.data_ptr(), batches, seq, heads, _ptr(kv_len), scale,
                                           _stream(qkv)), "f5_attention")
    return out


def row_norm(x: torch.Tensor, mode: int, a: torch.Tensor, b: Optional[torch.Tensor] = None, eps=1e-6) -> torch.Tensor:
    _need_cuda(x, a, b)
    assert x.dtype == torch.float32 and x.is_contiguous()
    rows, D = x.shape
    out = torch.empty((rows, D), dtype=torch.float16, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().f5_row_norm(x.data_ptr(), out.data_ptr(), rows, D, mode, eps, a.data_ptr(), _ptr(b),
                                          _stream(x)), "f5_row_norm")
    return out


def rope_tables(seq: int, device, dim_head=64):
    """fp32 cos/sin [seq, dim_head/2] of pos * 10000^(-2i/dim_head) (x_transformers RotaryEmbedding)"""
    inv = 1.0 / (10000 ** (torch.arange(0, dim_head, 2).float() / dim_head))
    ang = torch.outer(torch.arange(seq).float(), inv)
    return ang.cos().contiguous().to(device), ang.sin().contiguous().to(device)
