"""Tensor-level wrappers around the C ABI (include/llamax_b200.h).

PyTorch is used here only for device memory and streams: every function takes CUDA tensors, passes raw pointers,
sizes and the current stream to the library, and returns freshly allocated outputs. Nothing in this file computes
on the host and nothing falls back to PyTorch math.
"""

import ctypes
import threading

import torch
from torch import Tensor

from . import _lib
from ._lib import Epilogue, check

_tls = threading.local()


class _KernelTiming:
    """Optional CUDA-event timing of every library launch, by kernel class (used by bench.py for the live
    per-kernel roofline). Off by default: zero overhead on the training path."""

    def __init__(self):
        self.on = False
        self.only = None
        self.records = []

    def enable(self, only=None):
        """only: optional set of kernel classes to time (the others run without event records)."""
        self.records, self.on, self.only = [], True, (set(only) if only else None)

    def disable(self):
        self.on = False

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1, flops, nbytes in self.records:
            d = out.setdefault(name, {"ms": 0.0, "n": 0, "flops": 0.0, "bytes": 0.0})
            d["ms"] += e0.elapsed_time(e1)
            d["n"] += 1
            d["flops"] += flops
            d["bytes"] += nbytes
        return out


TIMING = _KernelTiming()


def _call(lib, name: str, args: tuple, kclass: str, flops: float = 0.0, nbytes: float = 0.0, shape=None):
    """Invoke one C-ABI entry point; raise on a non-zero return; optionally time it with CUDA events."""
    fn = getattr(lib, name)
    if TIMING.on and (TIMING.only is None or kclass in TIMING.only):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        TIMING.records.append((kclass, e0, e1, flops, nbytes))
        if shape is not None:
            TIMING.records.append((f"{kclass}[M={shape[0]},N={shape[1]},K={shape[2]}]", e0, e1, flops, nbytes))
    else:
        rc = fn(*args)
    check(rc, name)


def _prep(t: Tensor):
    """Select the tensor's device for this thread, return (lib, stream handle)."""
    if not t.is_cuda:
        raise _lib.LlamaxError("llamax_b200 ops need CUDA tensors: there is no CPU implementation of this path")
    lib = _lib.load()
    dev = t.device.index
    # always (re)select: torch.cuda.set_device / device guards on this thread may have changed the runtime's current
    # device since the last call, and a per-thread memo of "the device I selected last" cannot see that
    check(lib.llamax_set_device(dev), "llamax_set_device")
    return lib, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _rows(t: Tensor) -> Tensor:
    """View as 2-D [rows, last] with unit inner stride."""
    if t.dim() != 2:
        t = t.reshape(-1, t.shape[-1])
    if t.stride(1) != 1:
        t = t.contiguous()
    return t


def make_epilogue(lora_h=None, lora_b=None, lora_scale=1.0, resid=None, lora_seg=None, rope=None):
    """lora_seg = (n0, n1): three column segments [0, n0), [n0, n1), [n1, N) that use LoRA-h columns [0, R), [R, 2R),
    [2R, 3R) (lora_h is [M, 3R], lora_b the row-concatenated [N, R]) — q | k | v in one launch.
    rope = (table fp32 [S, 64, 2], S, rope_cols): RoPE on output columns [0, rope_cols) in the INT8 GEMM's epilogue."""
    if lora_h is None and resid is None and rope is None:
        return None, ()
    ep = Epilogue()
    keep = []
    if lora_h is not None:
        lora_h = _rows(lora_h)
        lora_b = lora_b.contiguous()
        assert lora_h.dtype is torch.bfloat16 and lora_b.dtype is torch.bfloat16
        rank = lora_b.shape[1]
        if lora_seg is not None:
            assert lora_h.shape[1] == 3 * rank and lora_seg[0] % 256 == 0 and lora_seg[1] % 256 == 0
            assert 0 < lora_seg[0] < lora_seg[1]
            ep.seg_n0, ep.seg_n1 = int(lora_seg[0]), int(lora_seg[1])
        else:
            assert rank == lora_h.shape[1]
        ep.lora_h, ep.ldh = lora_h.data_ptr(), lora_h.stride(0)
        ep.lora_b, ep.lora_rank, ep.lora_scale = lora_b.data_ptr(), rank, float(lora_scale)
        keep += [lora_h, lora_b]
    if resid is not None:
        resid = _rows(resid)
        assert resid.dtype is torch.bfloat16
        ep.resid, ep.ldr = resid.data_ptr(), resid.stride(0)
        keep.append(resid)
    if rope is not None:
        table, S, cols = rope
        assert table.dtype is torch.float32 and table.is_contiguous() and table.shape[0] >= S and table.shape[1:] == (64, 2)
        ep.rope, ep.rope_S, ep.rope_cols = table.data_ptr(), int(S), int(cols)
        keep.append(table)
    return ep, keep


def deterministic_mode(deterministic: bool | None = None) -> bool:
    """Whether a launch takes its deterministic form: `deterministic` when given, else PyTorch's own switch
    (torch.use_deterministic_algorithms). Deterministic forms give bitwise identical results from run to run on the same
    GPU: no fp32 reduction whose order depends on which CTA finishes first."""
    return torch.are_deterministic_algorithms_enabled() if deterministic is None else bool(deterministic)


def set_gemm_cta_group(cg: int):
    check(_lib.load().llamax_set_gemm_cta_group(cg), "llamax_set_gemm_cta_group")


# ---------------------------------------------------------------------------------------------- GEMMs
def int8_gemm_dequant(A: Tensor, W: Tensor, a_scale: Tensor, w_scale: Tensor, *, out: Tensor | None = None,
                      lora_h=None, lora_b=None, lora_scale=1.0, resid=None, lora_seg=None, rope=None) -> Tensor:
    """C = dequant(A[M,K] @ W[N,K]^T) (+ LoRA + residual). A, W int8; scales bf16.
    rope = (table, S, rope_cols): apply_rope on output columns [0, rope_cols) in the epilogue (head_dim 128)."""
    lib, st = _prep(A)
    assert A.dtype is torch.int8 and W.dtype is torch.int8 and A.dim() == 2 and W.dim() == 2
    assert A.stride(1) == 1 and W.stride(1) == 1 and A.shape[1] == W.shape[1]
    M, K = A.shape
    N = W.shape[0]
    a_scale = a_scale.reshape(-1).contiguous()
    w_scale = w_scale.reshape(-1).contiguous()
    assert a_scale.dtype is torch.bfloat16 and w_scale.dtype is torch.bfloat16
    assert a_scale.numel() == M and w_scale.numel() == N
    if out is None:
        out = torch.empty(M, N, device=A.device, dtype=torch.bfloat16)
    assert out.dtype is torch.bfloat16 and out.shape == (M, N) and out.stride(1) == 1
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, resid, lora_seg, rope)
    _call(lib, "llamax_int8_gemm_dequant",
          (_p(A), A.stride(0), _p(W), W.stride(0), _p(a_scale), _p(w_scale), _p(out), out.stride(0), M, N, K, ctypes.byref(ep) if ep is not None else None, st,),
          "int8_gemm", 2.0 * M * N * K, 0.0, shape=(M, N, K))
    return out


def int8_gemm_s32(A: Tensor, W: Tensor) -> Tensor:
    """Raw int32 accumulators of A[M,K] @ W[N,K]^T (parity/debug)."""
    lib, st = _prep(A)
    assert A.dtype is torch.int8 and W.dtype is torch.int8 and A.stride(1) == 1 and W.stride(1) == 1
    M, K = A.shape
    N = W.shape[0]
    out = torch.empty(M, N, device=A.device, dtype=torch.int32)
    _call(lib, "llamax_int8_gemm_s32",
          (_p(A), A.stride(0), _p(W), W.stride(0), _p(out), out.stride(0), M, N, K, st,),
          "int8_gemm", 2.0 * M * N * K, 0.0)
    return out


def bf16_gemm(A: Tensor, B: Tensor, *, col_scale: Tensor | None = None, round_before_scale: bool = False,
              out: Tensor | None = None, lora_h=None, lora_b=None, lora_scale=1.0, resid=None) -> Tensor:
    """C = A[M,K] @ B[N,K]^T (* col_scale) (+ LoRA + residual); bf16 in/out, fp32 accumulate."""
    lib, st = _prep(A)
    assert A.dtype is torch.bfloat16 and B.dtype is torch.bfloat16 and A.dim() == 2 and B.dim() == 2
    assert A.stride(1) == 1 and B.stride(1) == 1 and A.shape[1] == B.shape[1]
    M, K = A.shape
    N = B.shape[0]
    if col_scale is not None:
        col_scale = col_scale.reshape(-1).contiguous()
        assert col_scale.dtype is torch.bfloat16 and col_scale.numel() == N
    if out is None:
        out = torch.empty(M, N, device=A.device, dtype=torch.bfloat16)
    assert out.dtype is torch.bfloat16 and out.shape == (M, N) and out.stride(1) == 1
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, resid)
    _call(lib, "llamax_bf16_gemm",
          (_p(A), A.stride(0), _p(B), B.stride(0), _p(out), out.stride(0), M, N, K, _p(col_scale), int(round_before_scale), ctypes.byref(ep) if ep is not None else None, st,),
          "bf16_gemm", 2.0 * M * N * K, 0.0, shape=(M, N, K))
    return out


def bf16_gemm_swiglu_bwd(A: Tensor, B: Tensor, a: Tensor, b: Tensor, *, out_ab: Tensor, want_g: bool = False,
                         lora_h=None, lora_b=None, lora_scale=1.0):
    """swiglu_bwd(bf16(A[M,K] @ B[F,K]^T + LoRA term), a, b) with the SwiGLU backward as the GEMM's epilogue: the
    [M, F] gradient dg is never written. a, b: the two F-wide column blocks of one [M, >= 2F] buffer; da | db go to the
    first two F-wide column blocks of out_ab. Returns (da, db, g | None), identical to bf16_gemm -> swiglu_bwd."""
    lib, st = _prep(A)
    assert A.dtype is torch.bfloat16 and B.dtype is torch.bfloat16 and A.dim() == 2 and B.dim() == 2
    assert A.stride(1) == 1 and B.stride(1) == 1 and A.shape[1] == B.shape[1]
    M, K = A.shape
    F = B.shape[0]
    assert a.shape == (M, F) and b.shape == (M, F) and a.stride(1) == 1 and a.stride(0) == b.stride(0)
    assert b.data_ptr() == a.data_ptr() + 2 * F, "a | b must be adjacent column blocks of one buffer"
    assert out_ab.dtype is torch.bfloat16 and out_ab.shape[0] == M and out_ab.shape[1] >= 2 * F and out_ab.stride(1) == 1
    g = torch.empty(M, F, device=A.device, dtype=torch.bfloat16) if want_g else None
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, None)
    _call(lib, "llamax_bf16_gemm_swiglu_bwd",
          (_p(A), A.stride(0), _p(B), B.stride(0), M, F, K, ctypes.byref(ep) if ep is not None else None,
           _p(a), a.stride(0), _p(out_ab), out_ab.stride(0), _p(g), st,),
          "bf16_gemm", 2.0 * M * F * K, 0.0, shape=(M, F, K))
    return out_ab[:, :F], out_ab[:, F : 2 * F], g


def bf16_gemm_rowdot(A: Tensor, B: Tensor, other: Tensor, S: int, *, lora_h=None, lora_b=None, lora_scale=1.0):
    """C = A[M,K] @ B[N,K]^T (+ LoRA) and dot[b, g, s] = sum over the 128 columns of group g of C[b*S + s, c] * other[...]
    (C rounded to bf16 first): with other = the attention output this is the attention backward's delta, produced by the
    epilogue that writes dO. Returns (C, dot fp32 [M / S, N / 128, S])."""
    lib, st = _prep(A)
    assert A.dtype is torch.bfloat16 and B.dtype is torch.bfloat16 and other.dtype is torch.bfloat16
    assert A.dim() == 2 and B.dim() == 2 and A.stride(1) == 1 and B.stride(1) == 1 and A.shape[1] == B.shape[1]
    M, K = A.shape
    N = B.shape[0]
    other = _rows(other)
    assert other.shape == (M, N) and M % S == 0 and N % 256 == 0
    out = torch.empty(M, N, device=A.device, dtype=torch.bfloat16)
    dot = torch.empty(M // S, N // 128, S, device=A.device, dtype=torch.float32)
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, None)
    _call(lib, "llamax_bf16_gemm_rowdot",
          (_p(A), A.stride(0), _p(B), B.stride(0), _p(out), out.stride(0), M, N, K, ctypes.byref(ep) if ep is not None else None,
           _p(other), other.stride(0), _p(dot), S, st,),
          "bf16_gemm", 2.0 * M * N * K, 0.0, shape=(M, N, K))
    return out, dot


def bf16_int8_gemm(A: Tensor, W8: Tensor, w_scale: Tensor, *, out: Tensor | None = None, lora_h=None, lora_b=None,
                   lora_scale=1.0, resid=None) -> Tensor:
    """Weight-only forward, mixed-input (subclasses/int8.py:118): C = bf16(A[M,K] @ bf16(W8[N,K])^T) * w_scale[n]
    (+ LoRA + residual). The int8 weight is expanded to bf16 inside the GEMM's shared-memory pipeline: no de-quantised
    copy of W exists in HBM. Same arithmetic (and bits) as dequant_weight + bf16_gemm(round_before_scale=True)."""
    lib, st = _prep(A)
    assert A.dtype is torch.bfloat16 and W8.dtype is torch.int8 and A.dim() == 2 and W8.dim() == 2
    assert A.stride(1) == 1 and W8.stride(1) == 1 and A.shape[1] == W8.shape[1]
    M, K = A.shape
    N = W8.shape[0]
    w_scale = w_scale.reshape(-1).contiguous()
    assert w_scale.dtype is torch.bfloat16 and w_scale.numel() == N
    if out is None:
        out = torch.empty(M, N, device=A.device, dtype=torch.bfloat16)
    assert out.dtype is torch.bfloat16 and out.shape == (M, N) and out.stride(1) == 1
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, resid)
    _call(lib, "llamax_bf16_int8_gemm",
          (_p(A), A.stride(0), _p(W8), W8.stride(0), _p(w_scale), 0, None, 0, _p(out), out.stride(0), M, N, K, K,
           ctypes.byref(ep) if ep is not None else None, st,),
          "bf16_gemm", 2.0 * M * N * K, 0.0, shape=(M, N, K))
    return out


def _mixed_bwd_operands(A: Tensor, W8: Tensor, k_scale: Tensor, tail):
    assert A.dtype is torch.bfloat16 and W8.dtype is torch.int8 and A.dim() == 2 and W8.dim() == 2
    assert A.stride(1) == 1 and W8.stride(1) == 1
    K1, N = W8.shape
    k_scale = k_scale.reshape(-1).contiguous()
    assert k_scale.dtype is torch.bfloat16 and k_scale.numel() == K1
    rt = 0
    if tail is not None:
        assert tail.dtype is torch.bfloat16 and tail.dim() == 2 and tail.stride(1) == 1 and tail.shape[1] == N
        rt = tail.shape[0]
    assert A.shape[1] == K1 + rt, "A must be [M, K1 + tail rows]"
    return K1, N, rt, k_scale


def bf16_int8_gemm_bwd(A: Tensor, W8: Tensor, k_scale: Tensor, *, tail: Tensor | None = None, out: Tensor | None = None,
                       lora_h=None, lora_b=None, lora_scale=1.0) -> Tensor:
    """grad_input, mixed-input (subclasses/int8.py:127): C[M,N] = A[:, :K1] @ (k_scale[:, None] * W8[K1,N]) (+ A[:, K1:]
    @ tail[K-K1, N]) (+ LoRA epilogue). W8 is the frozen weight AS STORED ([out_features, in_features]: the contraction
    runs over out_features), or row-concatenated weights that share their input; tail = the LoRA A rows whose dh columns
    follow the gradient blocks in A. Bit-identical to bf16_gemm(A, [dequant_weight(W8, k_scale, transpose, scale) | tail^T])."""
    lib, st = _prep(A)
    K1, N, rt, k_scale = _mixed_bwd_operands(A, W8, k_scale, tail)
    M, K = A.shape
    if out is None:
        out = torch.empty(M, N, device=A.device, dtype=torch.bfloat16)
    assert out.dtype is torch.bfloat16 and out.shape == (M, N) and out.stride(1) == 1
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, None)
    _call(lib, "llamax_bf16_int8_gemm",
          (_p(A), A.stride(0), _p(W8), W8.stride(0), _p(k_scale), 1, _p(tail), tail.stride(0) if tail is not None else 0,
           _p(out), out.stride(0), M, N, K, K1, ctypes.byref(ep) if ep is not None else None, st,),
          "bf16_gemm", 2.0 * M * N * K, 0.0, shape=(M, N, K))
    return out


def bf16_int8_gemm_swiglu_bwd(A: Tensor, W8: Tensor, k_scale: Tensor, a: Tensor, b: Tensor, *, out_ab: Tensor,
                              want_g: bool = False, lora_h=None, lora_b=None, lora_scale=1.0):
    """bf16_gemm_swiglu_bwd with the mixed-input B operand of bf16_int8_gemm_bwd (W8 = w2 as stored, [D, F])."""
    lib, st = _prep(A)
    K1, F, rt, k_scale = _mixed_bwd_operands(A, W8, k_scale, None)
    M, K = A.shape
    assert a.shape == (M, F) and b.shape == (M, F) and a.stride(1) == 1 and a.stride(0) == b.stride(0)
    assert b.data_ptr() == a.data_ptr() + 2 * F, "a | b must be adjacent column blocks of one buffer"
    assert out_ab.dtype is torch.bfloat16 and out_ab.shape[0] == M and out_ab.shape[1] >= 2 * F and out_ab.stride(1) == 1
    g = torch.empty(M, F, device=A.device, dtype=torch.bfloat16) if want_g else None
    ep, keep = make_epilogue(lora_h, lora_b, lora_scale, None)
    _call(lib, "llamax_bf16_int8_gemm_swiglu_bwd",
          (_p(A), A.stride(0), _p(W8), W8.stride(0), _p(k_scale), M, F, K, ctypes.byref(ep) if ep is not None else None,
           _p(a), a.stride(0), _p(out_ab), out_ab.stride(0), _p(g), st,),
          "bf16_gemm", 2.0 * M * F * K, 0.0, shape=(M, F, K))
    return out_ab[:, :F], out_ab[:, F : 2 * F], g


def bf16_gemm_tn(At: Tensor, Bt: Tensor, *, out: Tensor | None = None) -> Tensor:
    """C[M,N] = At[K,M]^T @ Bt[K,N] (bf16 in/out, fp32 accumulate): the weight-gradient form, both operands consumed as
    stored (rows = the contraction index; row pitches may be smaller than the row length, i.e. overlapping rows)."""
    lib, st = _prep(At)
    assert At.dtype is torch.bfloat16 and Bt.dtype is torch.bfloat16 and At.dim() == 2 and Bt.dim() == 2
    assert At.stride(1) == 1 and Bt.stride(1) == 1 and At.shape[0] == Bt.shape[0]
    K, M = At.shape
    N = Bt.shape[1]
    if out is None:
        out = torch.empty(M, N, device=At.device, dtype=torch.bfloat16)
    assert out.dtype is torch.bfloat16 and out.shape == (M, N) and out.stride(1) == 1
    _call(lib, "llamax_bf16_gemm_tn",
          (_p(At), At.stride(0), _p(Bt), Bt.stride(0), _p(out), out.stride(0), M, N, K, st,),
          "bf16_gemm", 2.0 * M * N * K, 0.0, shape=(M, N, K))
    return out


def dequant_weight(w8: Tensor, scale: Tensor | None, *, transpose: bool, apply_scale: bool,
                   out: Tensor | None = None) -> Tensor:
    lib, st = _prep(w8)
    assert w8.dtype is torch.int8 and w8.is_contiguous()
    N, K = w8.shape
    shape = (K, N) if transpose else (N, K)
    if out is None:
        out = torch.empty(shape, device=w8.device, dtype=torch.bfloat16)
    assert out.shape == shape and out.stride(1) == 1 and out.dtype is torch.bfloat16
    if apply_scale:
        scale = scale.contiguous()
        assert scale.dtype is torch.bfloat16
    _call(lib, "llamax_dequant_weight",
          (_p(w8), _p(scale) if apply_scale else None, _p(out), out.stride(0), N, K, int(transpose), int(apply_scale), st,),
          "dequant_weight", 0.0, 3.0 * N * K)
    return out


# ------------------------------------------------------------------------------------------ elementwise
def rowquant_int8(x: Tensor):
    """quantize_int8_rowwise (subclasses/int8.py:10-16): returns (int8 [M,K], bf16 scale [M])."""
    x2 = _rows(x)
    lib, st = _prep(x2)
    assert x2.dtype is torch.bfloat16
    M, K = x2.shape
    q = torch.empty(M, K, device=x.device, dtype=torch.int8)
    s = torch.empty(M, device=x.device, dtype=torch.bfloat16)
    _call(lib, "llamax_rowquant_int8",
          (_p(x2), x2.stride(0), _p(q), _p(s), M, K, st,),
          "rowquant", 0.0, 3.0 * M * K)
    return q, s


def rowquant_int8_colscale(x: Tensor, col_scale: Tensor):
    """rowquant_int8 of x[m,c] * col_scale[c] (opt-in INT8 grad_input mode): returns (int8 [M,K], bf16 scale [M])."""
    x2 = _rows(x)
    lib, st = _prep(x2)
    assert x2.dtype is torch.bfloat16 and col_scale.dtype is torch.bfloat16 and col_scale.is_contiguous()
    M, K = x2.shape
    assert col_scale.numel() == K
    q = torch.empty(M, K, device=x.device, dtype=torch.int8)
    s = torch.empty(M, device=x.device, dtype=torch.bfloat16)
    _call(lib, "llamax_rowquant_int8_colscale",
          (_p(x2), x2.stride(0), _p(col_scale), _p(q), _p(s), M, K, st,),
          "rowquant", 0.0, 3.0 * M * K)
    return q, s


def rmsnorm_fwd(x: Tensor, w: Tensor, eps: float, *, quant: bool = False, want_y: bool = True):
    """Returns (y bf16 | None, rstd fp32 [M], q8 | None, qscale | None)."""
    x2 = _rows(x)
    assert x2.is_contiguous() and x2.dtype is torch.bfloat16 and w.dtype is torch.bfloat16 and w.is_contiguous()
    lib, st = _prep(x2)
    M, D = x2.shape
    y = torch.empty_like(x2) if want_y else None
    rstd = torch.empty(M, device=x.device, dtype=torch.float32)
    q8 = torch.empty(M, D, device=x.device, dtype=torch.int8) if quant else None
    qs = torch.empty(M, device=x.device, dtype=torch.bfloat16) if quant else None
    _call(lib, "llamax_rmsnorm_fwd",
          (_p(x2), _p(w), _p(y), _p(rstd), _p(q8), _p(qs), M, D, float(eps), st,),
          "rmsnorm_fwd", 0.0, (2.0 + 2.0 * (y is not None) + 1.0 * (q8 is not None)) * M * D)
    return y, rstd, q8, qs


def rmsnorm_bwd(dy: Tensor, x: Tensor, w: Tensor, rstd: Tensor, dres: Tensor | None, *, want_dw: bool = True):
    """Returns (dx bf16 [M,D], dw bf16 [D] | None). dx = dres + d(rmsnorm)/dx."""
    dy2, x2 = _rows(dy), _rows(x)
    assert dy2.is_contiguous() and x2.is_contiguous()
    lib, st = _prep(x2)
    M, D = x2.shape
    dres2 = None
    if dres is not None:
        dres2 = _rows(dres)
        assert dres2.is_contiguous()
    dx = torch.empty_like(x2)
    # two persistent CTAs per SM (the ring kernel's residency): one wave, no re-ramp of the prefetch rings
    nparts = max(1, min(int(M), 2 * torch.cuda.get_device_properties(x.device).multi_processor_count))
    partial = torch.empty(nparts, D, device=x.device, dtype=torch.float32) if want_dw else None
    _call(lib, "llamax_rmsnorm_bwd",
          (_p(dy2), _p(x2), _p(w), _p(rstd), _p(dres2), _p(dx), _p(partial), nparts, M, D, st,),
          "rmsnorm_bwd", 0.0, (6.0 + 2.0 * (dres2 is not None)) * M * D)
    dw = None
    if want_dw:
        dw = torch.empty(D, device=x.device, dtype=torch.bfloat16)
        _call(lib, "llamax_reduce_partials",
          (_p(partial), _p(dw), nparts, D, st,),
          "rmsnorm_bwd", 0.0, 4.0 * nparts * D)
    return dx, dw


def swiglu_fwd(a: Tensor, b: Tensor, *, quant: bool = False, want_g: bool = True):
    """g = bf16(bf16(silu(a)) * b). a, b: [M,F] views with a common row pitch. Returns (g, q8, qscale)."""
    lib, st = _prep(a)
    assert a.dtype is torch.bfloat16 and a.shape == b.shape and a.dim() == 2
    assert a.stride(1) == 1 and b.stride(1) == 1 and a.stride(0) == b.stride(0)
    M, F = a.shape
    g = torch.empty(M, F, device=a.device, dtype=torch.bfloat16) if want_g else None
    q8 = torch.empty(M, F, device=a.device, dtype=torch.int8) if quant else None
    qs = torch.empty(M, device=a.device, dtype=torch.bfloat16) if quant else None
    _call(lib, "llamax_swiglu_fwd",
          (_p(a), _p(b), a.stride(0), _p(g), _p(q8), _p(qs), M, F, st,),
          "swiglu_fwd", 0.0, (4.0 + 2.0 * (g is not None) + 1.0 * (q8 is not None)) * M * F)
    return g, q8, qs


def swiglu_bwd(dg: Tensor, a: Tensor, b: Tensor, *, want_g: bool = False, out_ab: Tensor | None = None):
    """Returns (da, db, g | None). If out_ab [M, >= 2F] is given, da/db are its first two F-wide column blocks."""
    lib, st = _prep(a)
    assert dg.is_contiguous() and a.stride(1) == 1 and a.stride(0) == b.stride(0)
    M, F = a.shape
    if out_ab is None:
        out_ab = torch.empty(M, 2 * F, device=a.device, dtype=torch.bfloat16)
    da, db = out_ab[:, :F], out_ab[:, F : 2 * F]
    g = torch.empty(M, F, device=a.device, dtype=torch.bfloat16) if want_g else None
    _call(lib, "llamax_swiglu_bwd",
          (_p(dg), _p(a), _p(b), a.stride(0), _p(da), _p(db), out_ab.stride(0), _p(g), M, F, st,),
          "swiglu_bwd", 0.0, (10.0 + 2.0 * (g is not None)) * M * F)
    return da, db, g


def rope_(x: Tensor, rope: Tensor, B: int, S: int, nheads: int, D: int, *, inverse: bool = False) -> Tensor:
    """In-place interleaved-pair RoPE on the first nheads*D columns of x [B*S, ld]."""
    lib, st = _prep(x)
    assert x.dtype is torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1 and x.shape[0] == B * S
    assert rope.dtype is torch.float32 and rope.is_contiguous() and rope.shape[0] >= S and rope.shape[1] == D // 2
    _call(lib, "llamax_rope_inplace",
          (_p(x), x.stride(0), _p(rope), B, S, nheads, D, int(inverse), st,),
          "rope", 0.0, 4.0 * B * S * nheads * D)
    return x


def transposed_rank_buffer(R: int, M: int, device) -> Tensor:
    """[R, M] bf16 buffer for an H^T operand: row pitch padded to a multiple of 8 elements (TMA), pad zeroed."""
    Mp = (M + 7) // 8 * 8
    if Mp == M:
        return torch.empty(R, M, device=device, dtype=torch.bfloat16)
    return torch.zeros(R, Mp, device=device, dtype=torch.bfloat16)[:, :M]


def lora_wgrad(X: Tensor, H: Tensor | None, alpha: float = 1.0, *, Ht: Tensor | None = None,
               deterministic: bool | None = None) -> Tensor:
    """out[P,R] (fp32) = alpha * X[M,P]^T @ H[M,R]  (tensor cores; X is consumed in place). Pass Ht = H^T [R,M]
    (from transposed_rank_buffer) when it already exists; otherwise it is made here (a tiny copy).
    deterministic (None: torch.are_deterministic_algorithms_enabled()): the token splits store partials into a
    workspace that is summed in split order, instead of fp32 atomics."""
    det = deterministic_mode(deterministic)
    lib, st = _prep(X)
    assert X.dtype is torch.bfloat16 and X.stride(1) == 1
    M, Pn = X.shape
    if Ht is None:
        assert H.dtype is torch.bfloat16
        Ht = transposed_rank_buffer(H.shape[1], M, X.device)
        Ht.copy_(H.t())
    R = Ht.shape[0]
    assert Ht.dtype is torch.bfloat16 and Ht.shape[1] == M and Ht.stride(1) == 1
    if R > 32:   # the kernel's accumulator is 32 columns wide: wider rank groups (e.g. q|k|v at rank 16) go in chunks
        return torch.cat([lora_wgrad(X, None, alpha, Ht=Ht[r0 : r0 + 32], deterministic=det) for r0 in range(0, R, 32)], 1)
    out = torch.empty(Pn, R, device=X.device, dtype=torch.float32)
    if det:
        ws = torch.empty(_lib.LORA_WGRAD_MAX_SPLITS, Pn, R, device=X.device, dtype=torch.float32)
        _call(lib, "llamax_lora_wgrad_deterministic",
              (_p(X), X.stride(0), _p(Ht), Ht.stride(0), _p(out), _p(ws), M, Pn, R, float(alpha), st),
              "lora_wgrad_det", 2.0 * M * Pn * R, 2.0 * M * (Pn + R))
        return out
    _call(lib, "llamax_lora_wgrad",
          (_p(X), X.stride(0), _p(Ht), Ht.stride(0), _p(out), M, Pn, R, float(alpha), st),
          "lora_wgrad", 2.0 * M * Pn * R, 2.0 * M * (Pn + R))
    return out


def lora_bwd_pair(dY: Tensor, Bt: Tensor, H: Tensor | None, out_dh: Tensor, alpha: float = 1.0, *,
                  Ht: Tensor | None = None, out_dht: Tensor | None = None) -> Tensor:
    """One pass over dY [M,N]: writes out_dh [M,R] = dY @ Bt^T (Bt = scale * B^T, [R,N]) and returns
    dB [N,R] (fp32) = alpha * dY^T @ H. Replaces a skinny dh GEMM + lora_wgrad that each streamed dY from HBM."""
    lib, st = _prep(dY)
    assert dY.dtype is torch.bfloat16 and Bt.dtype is torch.bfloat16
    assert dY.stride(1) == 1 and Bt.stride(1) == 1 and out_dh.stride(1) == 1 and out_dh.dtype is torch.bfloat16
    M, N = dY.shape
    if Ht is None:
        assert H.dtype is torch.bfloat16
        Ht = transposed_rank_buffer(H.shape[1], M, dY.device)
        Ht.copy_(H.t())
    R = Ht.shape[0]
    assert Ht.dtype is torch.bfloat16 and Ht.shape[1] == M and Ht.stride(1) == 1
    assert Bt.shape == (R, N) and out_dh.shape == (M, R)
    if out_dht is not None:   # also emit dh^T [R, M] (rows of a transposed_rank_buffer): the Ht operand of lora_wgrad
        assert out_dht.dtype is torch.bfloat16 and out_dht.shape == (R, M) and out_dht.stride(1) == 1
    dB = torch.empty(N, R, device=dY.device, dtype=torch.float32)
    acc = torch.empty(M, R, device=dY.device, dtype=torch.float32)
    _call(lib, "llamax_lora_bwd_pair",
          (_p(dY), dY.stride(0), _p(Bt), Bt.stride(0), _p(Ht), Ht.stride(0), _p(out_dh), out_dh.stride(0), _p(out_dht), out_dht.stride(0) if out_dht is not None else 0, _p(acc), _p(dB), M, N, R, float(alpha), st),
          "lora_wgrad", 4.0 * M * N * R, 2.0 * M * (N + 2 * R))
    return dB


def gelu_bias_fwd_(z: Tensor, bias: Tensor, period: int, lo: int, hi: int) -> Tensor:
    """In place z = bf16(z + bias); returns y = bf16(gelu_erf(z)). z: [rows, C] contiguous; rows whose index modulo
    `period` is outside [lo, hi) are padding rows and come out as zeros in both."""
    lib, st = _prep(z)
    assert z.dtype is torch.bfloat16 and z.dim() == 2 and z.is_contiguous() and bias.dtype is torch.bfloat16
    rows, C = z.shape
    y = torch.empty_like(z)
    _call(lib, "llamax_gelu_bias_fwd", (_p(z), _p(bias.contiguous()), _p(y), rows, C, period, lo, hi, st),
          "gelu", 0.0, 6.0 * rows * C)
    return y


def gelu_bwd(dy: Tensor, z: Tensor, period: int, lo: int, hi: int, out: Tensor | None = None) -> Tensor:
    """dz = bf16(dy * gelu_erf'(z)), zeros on padding rows."""
    lib, st = _prep(z)
    assert dy.dtype is torch.bfloat16 and dy.is_contiguous() and z.is_contiguous() and dy.shape == z.shape
    rows, C = z.shape
    dz = torch.empty_like(z) if out is None else out
    _call(lib, "llamax_gelu_bwd", (_p(dy), _p(z), _p(dz), rows, C, period, lo, hi, st), "gelu", 0.0, 6.0 * rows * C)
    return dz


def conv_s2k3_col2im(dcol: Tensor, B: int, Tp: int, C: int) -> Tensor:
    """dcol [B * Tp/2, 3C] (row t of a slab = gradients of padded input rows 2t..2t+2) -> dxp [B, Tp, C]."""
    lib, st = _prep(dcol)
    assert dcol.dtype is torch.bfloat16 and dcol.is_contiguous() and dcol.shape == (B * (Tp // 2), 3 * C)
    dxp = torch.empty(B, Tp, C, device=dcol.device, dtype=torch.bfloat16)
    _call(lib, "llamax_conv_s2k3_col2im", (_p(dcol), _p(dxp), B, Tp, C, st), "col2im", 0.0, 5.0 * B * Tp * C)
    return dxp


def batched_copy(jobs) -> None:
    """jobs: iterable of (src, dst, scale, transpose). dst (bf16, 2-D, unit inner stride) receives
    bf16(scale * src) or its transpose; src is a 2-D bf16 / fp32 tensor with unit inner stride. ONE launch per
    64 jobs instead of one elementwise launch (or three) per job."""
    jobs = list(jobs)
    if not jobs:
        return
    lib, st = _prep(jobs[0][0])
    for i0 in range(0, len(jobs), _lib.MAX_COPY_JOBS):
        chunk = jobs[i0 : i0 + _lib.MAX_COPY_JOBS]
        arr = (_lib.CopyJob * len(chunk))()
        for k, (src, dst, scale, transpose) in enumerate(chunk):
            assert src.dim() == 2 and dst.dim() == 2 and src.stride(1) == 1 and dst.stride(1) == 1
            assert dst.dtype is torch.bfloat16 and src.dtype in (torch.bfloat16, torch.float32)
            assert tuple(dst.shape) == ((src.shape[1], src.shape[0]) if transpose else tuple(src.shape))
            j = arr[k]
            j.src, j.dst = src.data_ptr(), dst.data_ptr()
            j.src_ld, j.dst_ld = src.stride(0), dst.stride(0)
            j.rows, j.cols = src.shape
            j.scale = float(scale)
            j.flags = (1 if src.dtype is torch.float32 else 0) | (2 if transpose else 0)
        _call(lib, "llamax_batched_copy", (arr, len(chunk), st), "batched_copy", 0.0, 0.0)


def cross_entropy_(logits: Tensor, labels: Tensor, loss_sum: Tensor, inv_n: Tensor | None, write_grad: bool, *,
                   deterministic: bool | None = None):
    """In place: accumulates sum of per-row CE into loss_sum (fp32 scalar tensor); if write_grad, overwrites logits
    with (softmax - onehot) * inv_n (rows with label -100 -> 0).
    deterministic (None: torch.are_deterministic_algorithms_enabled()): the row losses go to an fp32 [M] buffer and are
    summed in a fixed order, instead of fp32 atomics in CTA completion order."""
    lib, st = _prep(logits)
    assert logits.dtype is torch.bfloat16 and logits.dim() == 2 and logits.stride(1) == 1
    assert labels.dtype is torch.int64 and labels.is_contiguous() and labels.numel() == logits.shape[0]
    assert loss_sum.dtype is torch.float32 and (inv_n is None or inv_n.dtype is torch.float32)
    M, V = logits.shape
    if deterministic_mode(deterministic):
        rows = torch.empty(M, device=logits.device, dtype=torch.float32)
        _call(lib, "llamax_cross_entropy_rows",
              (_p(logits), logits.stride(0), _p(labels), _p(rows), _p(inv_n), M, V, int(write_grad), st),
              "cross_entropy_det", 0.0, (4.0 if write_grad else 2.0) * M * V)
        loss_sum += rows.sum()   # fixed-order tree reduction for a given M
        return
    _call(lib, "llamax_cross_entropy",
          (_p(logits), logits.stride(0), _p(labels), _p(loss_sum), _p(inv_n), M, V, int(write_grad), st),
          "cross_entropy", 0.0, (4.0 if write_grad else 2.0) * M * V)


# ---------------------------------------------------------------------------------------------- attention
def _pairs(S: int, prefix_len) -> float:
    """Unmasked (q, kv) pairs of the prefix-LM mask: S*P + (S-P)(S-P+1)/2 (mean over the batch for per-sequence P)."""
    if isinstance(prefix_len, Tensor):
        if not TIMING.on:
            return 0.0          # only the timing report needs it: no device sync on the training path
        return float(sum(_pairs(S, int(v)) for v in prefix_len.tolist())) / max(1, prefix_len.numel())
    P_ = min(int(prefix_len), S)
    return S * P_ + (S - P_) * (S - P_ + 1) / 2


def _prefix_args(prefix_len, B: int, device):
    """(scalar prefix, int32 [B] device pointer tensor | None) for the C ABI."""
    if isinstance(prefix_len, Tensor):
        pb = prefix_len.to(device=device, dtype=torch.int32).reshape(-1).contiguous()
        assert pb.numel() == B, f"per-sequence prefix_len must have {B} entries"
        return 0, pb
    return int(prefix_len), None


def doc_bounds(doc_ids: Tensor):
    """doc_ids int [B, S] (non-decreasing per row: packed documents) -> (doc_start, doc_end) int32 [B, S]."""
    B, S = doc_ids.shape
    idx = torch.arange(S, device=doc_ids.device).expand(B, S)
    first = torch.ones_like(doc_ids, dtype=torch.bool)
    first[:, 1:] = doc_ids[:, 1:] != doc_ids[:, :-1]
    last = torch.ones_like(first)
    last[:, :-1] = first[:, 1:]
    start = torch.where(first, idx, torch.zeros_like(idx)).cummax(dim=1).values
    end = torch.where(last, idx, torch.full_like(idx, S - 1)).flip(1).cummin(dim=1).values.flip(1)
    return start.to(torch.int32).contiguous(), end.to(torch.int32).contiguous()


def attn_fwd(q: Tensor, k: Tensor, v: Tensor, B: int, S: int, Hq: int, Hkv: int, D: int, prefix_len,
             scale: float | None = None, doc_start: Tensor | None = None):
    """q [B*S, Hq*D] / k, v [B*S, Hkv*D] row views (unit inner stride). prefix_len: int, or an int tensor [B] with one
    prefix length per sequence. Returns (o [B*S, Hq*D], lse [B,Hq,S])."""
    lib, st = _prep(q)
    for t in (q, k, v):
        assert t.dtype is torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1 and t.shape[0] == B * S
    o = torch.empty(B * S, Hq * D, device=q.device, dtype=torch.bfloat16)
    lse = torch.empty(B, Hq, S, device=q.device, dtype=torch.float32)
    scale = float(scale) if scale is not None else D ** -0.5
    p_scalar, p_b = _prefix_args(prefix_len, B, q.device)
    _call(lib, "llamax_attn_fwd",
          (_p(q), q.stride(0), _p(k), k.stride(0), _p(v), v.stride(0), _p(o), o.stride(0), _p(lse), B, S, Hq, Hkv, D, p_scalar, _p(p_b), _p(doc_start), scale, st,),
          "attn_fwd", 4.0 * B * Hq * D * _pairs(S, prefix_len), 0.0)
    return o, lse


def attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, B, S, Hq, Hkv, D, prefix_len, scale=None, doc_start=None,
             doc_end=None, rope_inverse=None, delta=None, *, deterministic: bool | None = None):
    """Writes dq/dk/dv (row views like q/k/v). rope_inverse: fp32 [>= S, D/2, 2] table -> dq, dk come back already
    rotated through the RoPE backward (no separate rope_(..., inverse=True) pass needed). delta: fp32 [B, Hq, S] =
    sum_d dout * o already computed (bf16_gemm_rowdot): o is then not read and may be None.
    deterministic (None: torch.are_deterministic_algorithms_enabled()): dq from a kernel that sums the kv tiles of each
    query tile in a fixed order (it recomputes the S and dP products) instead of fp32 atomics; dk, dv are unchanged."""
    det = deterministic_mode(deterministic)
    if rope_inverse is not None:
        assert rope_inverse.dtype is torch.float32 and rope_inverse.is_contiguous()
        assert rope_inverse.shape[0] >= S and rope_inverse.shape[1] == D // 2
    lib, st = _prep(q)
    dout = _rows(dout)
    dq_accum = None if det else torch.empty(B * S, Hq * D, device=q.device, dtype=torch.float32)
    if delta is None:
        delta = torch.empty(B, Hq, S, device=q.device, dtype=torch.float32)
    else:
        assert delta.dtype is torch.float32 and delta.shape == (B, Hq, S) and delta.is_contiguous()
        o = None
    scale = float(scale) if scale is not None else D ** -0.5
    p_scalar, p_b = _prefix_args(prefix_len, B, q.device)
    if det:
        _call(lib, "llamax_attn_bwd_deterministic",
              (_p(q), q.stride(0), _p(k), k.stride(0), _p(v), v.stride(0), _p(o), o.stride(0) if o is not None else 0, _p(lse), _p(dout), dout.stride(0), _p(dq), dq.stride(0), _p(dk), dk.stride(0), _p(dv), dv.stride(0), _p(delta), B, S, Hq, Hkv, D, p_scalar, _p(p_b), _p(doc_start), _p(doc_end), scale, _p(rope_inverse), st,),
              "attn_bwd_det", 14.0 * B * Hq * D * _pairs(S, prefix_len), 0.0)
        return dq, dk, dv
    _call(lib, "llamax_attn_bwd",
          (_p(q), q.stride(0), _p(k), k.stride(0), _p(v), v.stride(0), _p(o), o.stride(0) if o is not None else 0, _p(lse), _p(dout), dout.stride(0), _p(dq), dq.stride(0), _p(dk), dk.stride(0), _p(dv), dv.stride(0), _p(dq_accum), _p(delta), B, S, Hq, Hkv, D, p_scalar, _p(p_b), _p(doc_start), _p(doc_end), scale, _p(rope_inverse), st,),
          "attn_bwd", 10.0 * B * Hq * D * _pairs(S, prefix_len), 0.0)
    return dq, dk, dv
