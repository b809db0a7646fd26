"""CPU oracle for the llama-x fine-tuning hot path.  TEST INFRASTRUCTURE ONLY.

A plain-PyTorch (CPU) restatement of the reference algorithm for every function on the path, each citing the
reference file:line it follows (paths relative to the gau-nernst/llama-x repo).  Only `tests/`,
`__graft_entry__.smoke()` and the `cpu_baseline` / `--impl reference` legs of `bench.py` may import this package;
the product (`llamax_b200/`) never does.

Parity pin: the reference ships no tests or golden vectors (SURVEY.md §4), so this restatement is pinned against
outputs of the reference code itself, executed in the build container with fixed seeds
(`oracle/make_golden.py` -> `tests/golden/reference_vectors.pt.xz`; checked by `tests/test_oracle_golden.py`).

Two flavours are provided where rounding matters:
  * `*_ref`  : the reference's own bf16 op sequence (bit-comparable to the reference on CPU)
  * `*_f32`  : the same math evaluated in fp32 without intermediate rounding (tolerance checks)
"""

from __future__ import annotations

import math

import torch
import torch.nn.functional as F
from torch import Tensor

# ------------------------------------------------------------------------------------------------
# K2  row-wise int8 quantisation                                   subclasses/int8.py:10-16
# ------------------------------------------------------------------------------------------------
def quantize_int8_rowwise(x: Tensor):
    xf = x.to(torch.float32)
    s = xf.abs().amax(dim=1) / 127
    q = (xf / s.clamp_min(1e-12).unsqueeze(1)).round().to(torch.int8)
    return q, s.to(x.dtype)


# ------------------------------------------------------------------------------------------------
# K3  int8 GEMM + dequant                                           subclasses/int8_mm.py:93-118
# ------------------------------------------------------------------------------------------------
def int8_mm_s32(A: Tensor, B: Tensor) -> Tensor:
    """Exact int32 accumulators of A[M,K] @ B[K,N] (int8 operands)."""
    return A.to(torch.int32) @ B.to(torch.int32) if A.shape[0] < 17 else torch._int_mm(A, B)


def int8_mm_dequant(A: Tensor, B: Tensor, a_scale: Tensor, b_scale: Tensor) -> Tensor:
    acc = int8_mm_s32(A, B).to(torch.float32)
    out = (acc * a_scale.to(torch.float32).reshape(-1, 1)) * b_scale.to(torch.float32).reshape(1, -1)
    return out.to(a_scale.dtype)


# ------------------------------------------------------------------------------------------------
# a7/a9  _Int8Linear forward / backward                              subclasses/int8.py:107-130
# ------------------------------------------------------------------------------------------------
def int8_linear_fwd_ref(x: Tensor, w8: Tensor, w_scale: Tensor, dynamic_int8_act: bool) -> Tensor:
    if dynamic_int8_act:
        x8, xs = quantize_int8_rowwise(x.reshape(-1, w8.shape[1]))
        out = int8_mm_dequant(x8, w8.T, xs, w_scale)
        return out.reshape(*x.shape[:-1], -1)
    return (x @ w8.T.to(x.dtype)) * w_scale


def int8_linear_bwd_ref(grad_out: Tensor, w8: Tensor, w_scale: Tensor) -> Tensor:
    return (grad_out * w_scale) @ w8.to(grad_out.dtype)


def int8_linear_fwd_f32(x: Tensor, w8: Tensor, w_scale: Tensor) -> Tensor:
    """Ideal (unquantised-activation) value: x @ (s * W8)^T in fp32."""
    return x.float() @ (w8.float() * w_scale.float().unsqueeze(1)).T


def int8_linear_bwd_f32(grad_out: Tensor, w8: Tensor, w_scale: Tensor) -> Tensor:
    return grad_out.float() @ (w8.float() * w_scale.float().unsqueeze(1))


# ------------------------------------------------------------------------------------------------
# a4  LoRA                                                            modelling/lora.py:40-44
# ------------------------------------------------------------------------------------------------
def lora_delta_ref(x: Tensor, lora_a: Tensor, lora_b: Tensor, scale: float) -> Tensor:
    return x @ lora_a.T @ lora_b.T * scale


def lora_delta_f32(x: Tensor, lora_a: Tensor, lora_b: Tensor, scale: float) -> Tensor:
    return (x.float() @ lora_a.float().T) @ lora_b.float().T * scale


# ------------------------------------------------------------------------------------------------
# K1  RMSNorm                         nn.RMSNorm(dim, eps=1e-5) at modelling/llama.py:158,160,182
# ------------------------------------------------------------------------------------------------
def rmsnorm_ref(x: Tensor, w: Tensor, eps: float = 1e-5) -> Tensor:
    xf = x.float()
    y = xf * torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps) * w.float()
    return y.to(x.dtype)


def rmsnorm_bwd_f32(dy: Tensor, x: Tensor, w: Tensor, eps: float = 1e-5):
    xf, dyf, wf = x.float(), dy.float(), w.float()
    rstd = torch.rsqrt(xf.pow(2).mean(-1, keepdim=True) + eps)
    xhat = xf * rstd
    g = dyf * wf
    dx = rstd * (g - xhat * (g * xhat).mean(-1, keepdim=True))
    dw = (dyf * xhat).reshape(-1, x.shape[-1]).sum(0)
    return dx, dw


# ------------------------------------------------------------------------------------------------
# K10  SwiGLU                                                         modelling/llama.py:149,152
# ------------------------------------------------------------------------------------------------
def swiglu_ref(a: Tensor, b: Tensor) -> Tensor:
    return F.silu(a) * b


def swiglu_f32(a: Tensor, b: Tensor) -> Tensor:
    return F.silu(a.float()) * b.float()


def swiglu_bwd_f32(dg: Tensor, a: Tensor, b: Tensor):
    af, bf, dgf = a.float(), b.float(), dg.float()
    sig = torch.sigmoid(af)
    da = dgf * bf * sig * (1 + af * (1 - sig))
    db = dgf * af * sig
    return da, db


# ------------------------------------------------------------------------------------------------
# K7  RoPE                                                            modelling/llama.py:32-73
# ------------------------------------------------------------------------------------------------
def llama3_1_rescale(freqs: Tensor) -> Tensor:
    """Llama-3.1 frequency rescale (factor 8, low 1, high 4, original context 8192); llama.py:32-51."""
    factor, low, high, old_ctx = 8, 1, 4, 8192
    out = []
    for f in freqs:
        wavelen = 2 * torch.pi / f
        if wavelen < old_ctx / high:
            out.append(f)
        elif wavelen > old_ctx / low:
            out.append(f / factor)
        else:
            smooth = (old_ctx / wavelen - low) / (high - low)
            out.append((1 - smooth) * f / factor + smooth * f)
    return torch.tensor(out, dtype=freqs.dtype)


def build_rope(head_dim: int, max_seq_len: int, rope_base: float, is_llama3_1: bool) -> Tensor:
    """[max_seq_len, head_dim/2, 2] fp32 table of (cos, sin); llama.py:54-60."""
    theta = 1.0 / (rope_base ** (torch.arange(0, head_dim, 2, dtype=torch.float32) / head_dim))
    if is_llama3_1:
        theta = llama3_1_rescale(theta)
    ang = torch.outer(torch.arange(max_seq_len, dtype=torch.float32), theta)
    return torch.stack([ang.cos(), ang.sin()], dim=-1)


def apply_rope(x: Tensor, rope: Tensor) -> Tensor:
    """x [B, S, H, D]; rotates adjacent pairs (2i, 2i+1) in fp32; llama.py:63-73."""
    cs = rope.reshape(1, x.shape[1], 1, -1, 2)
    xp = x.float().unflatten(-1, (-1, 2))
    x0, x1 = xp[..., 0], xp[..., 1]
    y = torch.stack([x0 * cs[..., 0] - x1 * cs[..., 1], x1 * cs[..., 0] + x0 * cs[..., 1]], dim=-1)
    return y.flatten(3).to(x.dtype)


def apply_rope_inverse(dy: Tensor, rope: Tensor) -> Tensor:
    """Backward of apply_rope (rotation by -theta), fp32 math."""
    cs = rope.reshape(1, dy.shape[1], 1, -1, 2)
    dp = dy.float().unflatten(-1, (-1, 2))
    d0, d1 = dp[..., 0], dp[..., 1]
    dx = torch.stack([d0 * cs[..., 0] + d1 * cs[..., 1], d1 * cs[..., 0] - d0 * cs[..., 1]], dim=-1)
    return dx.flatten(3).to(dy.dtype)


# ------------------------------------------------------------------------------------------------
# K8/K9  attention with the prefix-LM mask                            modelling/llama.py:129-137
# ------------------------------------------------------------------------------------------------
def prefix_lm_mask(L: int, prefix_len: int) -> Tensor:
    """mask[q, kv] = (kv < P) | (q >= kv): bidirectional prefix, causal suffix (README.md:16 plan)."""
    q = torch.arange(L).unsqueeze(1)
    kv = torch.arange(L).unsqueeze(0)
    return (kv < prefix_len) | (q >= kv)


def document_causal_mask(doc_ids: Tensor) -> Tensor:
    """[B, 1, S, S] mask of the packed-sequence trainer: same document and causal (train_metamathqa.py:67-70)."""
    S = doc_ids.shape[-1]
    same = doc_ids[:, :, None] == doc_ids[:, None, :]
    return (same & torch.tril(torch.ones(S, S, dtype=torch.bool)))[:, None]


def attention_ref(q: Tensor, k: Tensor, v: Tensor, prefix_len: int, dtype=torch.float32, doc_ids=None) -> Tensor:
    """q [B,Hq,S,D], k/v [B,Hkv,S,D] -> [B,Hq,S,D]; dense masked softmax evaluated in `dtype`."""
    B, Hq, S, D = q.shape
    rep = Hq // k.shape[1]
    qf = q.to(dtype)
    kf = k.to(dtype).repeat_interleave(rep, dim=1)
    vf = v.to(dtype).repeat_interleave(rep, dim=1)
    s = (qf @ kf.transpose(-1, -2)) / math.sqrt(D)
    mask = prefix_lm_mask(S, prefix_len) if doc_ids is None else document_causal_mask(doc_ids)
    s = s.masked_fill(~mask, float("-inf"))
    return torch.softmax(s, dim=-1) @ vf


def attention_ref_grads(q, k, v, dout, prefix_len, dtype=torch.float64, doc_ids=None):
    """(out, dq, dk, dv) via autograd on the dense formulation in `dtype`."""
    q_, k_, v_ = (t.detach().to(dtype).requires_grad_(True) for t in (q, k, v))
    out = attention_ref(q_, k_, v_, prefix_len, dtype, doc_ids)
    out.backward(dout.to(dtype))
    return out.detach(), q_.grad, k_.grad, v_.grad


def attention_ref_grouped(q, k, v, dout, prefix_len, doc_ids=None, scale=None, delta_from_bf16_o=False):
    """The math of `attention_ref_grads` in fp64, written out and evaluated one (sequence, kv head) group at a time on
    the device of the inputs, so that it scales to full-size shapes on a GPU (fp64 matmuls ignore the TF32 flags).

    q, dout [B,Hq,S,D], k, v [B,Hkv,S,D] (any float dtype); prefix_len: int, or a sequence / tensor of B lengths;
    doc_ids: int [B, S] packed-document ids or None; scale: softmax scale (default D**-0.5).
    delta_from_bf16_o: take delta = rowsum(bf16(o) * dout) instead of rowsum(o * dout), i.e. the rounding a kernel that
    reads its own bf16 output for delta cannot avoid.
    Returns fp64 (o [B,Hq,S,D], lse [B,Hq,S] (natural log), dq [B,Hq,S,D], dk, dv [B,Hkv,S,D])."""
    B, Hq, S, D = q.shape
    Hkv = k.shape[1]
    G = Hq // Hkv
    scale = D ** -0.5 if scale is None else float(scale)
    dev, f64 = q.device, torch.float64
    prefix = [int(p) for p in prefix_len] if isinstance(prefix_len, (list, tuple, Tensor)) else [int(prefix_len)] * B
    o = torch.empty(B, Hq, S, D, dtype=f64, device=dev)
    lse = torch.empty(B, Hq, S, dtype=f64, device=dev)
    dq = torch.empty(B, Hq, S, D, dtype=f64, device=dev)
    dk = torch.empty(B, Hkv, S, D, dtype=f64, device=dev)
    dv = torch.empty(B, Hkv, S, D, dtype=f64, device=dev)
    idx = torch.arange(S, device=dev)
    for b in range(B):
        if doc_ids is None:
            mask = (idx[None, :] < prefix[b]) | (idx[:, None] >= idx[None, :])
        else:
            d = doc_ids[b].to(dev)
            mask = (d[:, None] == d[None, :]) & (idx[:, None] >= idx[None, :])
        for hk in range(Hkv):
            hs = slice(hk * G, (hk + 1) * G)
            qg, dog = q[b, hs].to(f64), dout[b, hs].to(f64)          # [G, S, D]
            kg, vg = k[b, hk].to(f64), v[b, hk].to(f64)              # [S, D]
            s = (qg @ kg.T) * scale
            s.masked_fill_(~mask, float("-inf"))
            m = s.amax(-1, keepdim=True)
            p = torch.exp(s - m)
            l = p.sum(-1, keepdim=True)
            p /= l
            og = p @ vg
            o[b, hs], lse[b, hs] = og, (m + l.log()).squeeze(-1)
            ob = og.to(torch.bfloat16).to(f64) if delta_from_bf16_o else og
            delta = (ob * dog).sum(-1, keepdim=True)
            ds = p * (dog @ vg.T - delta)                            # dS = P o (dP - delta), then dS * scale below
            dq[b, hs] = (ds @ kg) * scale
            dk[b, hk] = torch.einsum("gqk,gqd->kd", ds, qg) * scale
            dv[b, hk] = torch.einsum("gqk,gqd->kd", p, dog)
    return o, lse, dq, dk, dv


# ------------------------------------------------------------------------------------------------
# a1/a3/a12  decoder block                                            modelling/llama.py:93-174
# ------------------------------------------------------------------------------------------------
class LayerWeights:
    """Plain container: int8 weights + scales + LoRA factors + norm weights of one TransformerLayer."""

    names = ("wq", "wk", "wv", "wo", "w1", "w3", "w2")

    def __init__(self):
        self.w8 = {}
        self.ws = {}
        self.lora_a = {}
        self.lora_b = {}
        self.lora_scale = 1.0
        self.attention_norm = None
        self.ffn_norm = None


class Int8LinearRef(torch.autograd.Function):
    """The reference's custom autograd node (subclasses/int8.py:106-130): forward in either INT8 mode, backward
    grad_input = (grad * scale) @ W8 in the gradient's dtype — a straight-through estimator that ignores the
    activation quantisation of the dynamic mode; the frozen weight gets no gradient."""

    @staticmethod
    def forward(ctx, x, w8, w_scale, dynamic_int8_act):
        ctx.save_for_backward(w8, w_scale)
        return int8_linear_fwd_ref(x, w8, w_scale, dynamic_int8_act)

    @staticmethod
    def backward(ctx, grad_out):
        w8, w_scale = ctx.saved_tensors
        return int8_linear_bwd_ref(grad_out, w8, w_scale), None, None, None


def lora_linear_ref(x, lw: LayerWeights, name: str, dynamic: bool):
    out = Int8LinearRef.apply(x, lw.w8[name], lw.ws[name], dynamic)
    if name in lw.lora_a:
        out = out + lora_delta_ref(x, lw.lora_a[name], lw.lora_b[name], lw.lora_scale)
    return out


def transformer_layer_ref(x: Tensor, rope: Tensor, lw: LayerWeights, Hq: int, Hkv: int, D: int, prefix_len: int,
                          dynamic: bool, doc_ids: Tensor | None = None) -> Tensor:
    """Reference op sequence of TransformerLayer.forward (llama.py:163-174) in the input dtype (bf16)."""
    B, L, _ = x.shape
    h = rmsnorm_ref(x, lw.attention_norm)
    q = lora_linear_ref(h, lw, "wq", dynamic).view(B, L, Hq, D)
    k = lora_linear_ref(h, lw, "wk", dynamic).view(B, L, Hkv, D)
    v = lora_linear_ref(h, lw, "wv", dynamic).view(B, L, Hkv, D)
    q = apply_rope(q, rope).transpose(1, 2)
    k = apply_rope(k, rope).transpose(1, 2)
    v = v.transpose(1, 2)
    mask = prefix_lm_mask(L, prefix_len) if doc_ids is None else document_causal_mask(doc_ids)
    o = F.scaled_dot_product_attention(q, k, v, mask, 0.0, False, enable_gqa=True)
    o = o.transpose(1, 2).reshape(B, L, Hq * D)
    x = x + lora_linear_ref(o, lw, "wo", dynamic)
    h = rmsnorm_ref(x, lw.ffn_norm)
    g = swiglu_ref(lora_linear_ref(h, lw, "w1", dynamic), lora_linear_ref(h, lw, "w3", dynamic))
    return x + lora_linear_ref(g, lw, "w2", dynamic)


def audio_stem_ref(mel: Tensor, w1: Tensor, b1: Tensor, w2: Tensor, b2: Tensor) -> Tensor:
    """Whisper-style stem of LlamaAudio (modelling/audio.py:26-31 applied at :56-60), evaluated in the dtype of its
    inputs: GELU(Conv1d(k3, s2, p1)(GELU(Conv1d(k3, s1, p1)(mel)))).transpose(1, 2).  mel [B, n_mels, T]."""
    x = F.gelu(F.conv1d(mel, w1, b1, stride=1, padding=1))
    x = F.gelu(F.conv1d(x, w2, b2, stride=2, padding=1))
    return x.transpose(1, 2)
