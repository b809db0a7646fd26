"""Reference of the attention dropout of the attention kernels (include/llamax_b200.h, llamax_attn_*_dropout).
TEST INFRASTRUCTURE ONLY, like oracle/ref_ops.py, whose building blocks it reuses.

  * `philox4x32_10`: Philox4x32-10 (Random123 / curand) in numpy;
  * `attention_dropout_keep`: the keep mask Z the kernels regenerate from (seed, offset);
  * `attention_ref_grouped_dropout`: oracle/ref_ops.attention_ref_grouped's fp64 math with Z applied;
  * `transformer_layer_ref_dropout`: oracle/ref_ops.transformer_layer_ref with Z applied to the attention probabilities.
"""
from __future__ import annotations

import numpy as np
import torch
from torch import Tensor

from oracle import ref_ops as R

_PHILOX_M = (0xD2511F53, 0xCD9E8D57)
_PHILOX_W = (0x9E3779B9, 0xBB67AE85)


def philox4x32_10(ctr, key) -> np.ndarray:
    """Philox4x32-10 (Random123 / curand): ctr uint32 [..., 4], key uint32 [..., 2] (broadcast) -> uint32 [..., 4]."""
    m32 = np.uint64(0xFFFFFFFF)
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] for i in range(4)]
    k = [np.asarray(key, dtype=np.uint64)[..., i] for i in range(2)]
    for r in range(10):
        if r:
            k = [(k[0] + np.uint64(_PHILOX_W[0])) & m32, (k[1] + np.uint64(_PHILOX_W[1])) & m32]
        p0, p1 = np.uint64(_PHILOX_M[0]) * c[0], np.uint64(_PHILOX_M[1]) * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & m32, p1 >> np.uint64(32), p1 & m32
        c = [hi1 ^ c[1] ^ k[0], lo1, hi0 ^ c[3] ^ k[1], lo0]
    return np.stack(c, -1).astype(np.uint32)


def attention_dropout_threshold(p: float) -> tuple[int, float]:
    """(t, scale): a key is kept when its Philox byte is >= t = round(256 p); kept values are scaled by 256 / (256 - t)
    (0 when t = 256: everything is dropped). The drop rate is exactly t / 256."""
    t = int(round(p * 256))
    return t, (0.0 if t >= 256 else 256.0 / (256 - t))


def attention_dropout_keep(seed: int, offset: int, B: int, Hq: int, S: int, p: float, *, q_start: int = 0,
                           q_len: int | None = None, kv_start: int = 0, kv_len: int | None = None) -> Tensor:
    """Keep mask Z (bool [B, Hq, q_len, kv_len]): key = the 64-bit seed, counter = (kv // 16, q, b * Hq + hq,
    offset // 4), key kv kept when byte kv % 16 of the output (little-endian) is >= t. The window
    [q_start, +q_len) x [kv_start, +kv_len) (default: all of S x S) limits the work for long sequences."""
    q_len = S - q_start if q_len is None else q_len
    kv_len = S - kv_start if kv_len is None else kv_len
    t, _ = attention_dropout_threshold(p)
    g0, g1 = kv_start // 16, (kv_start + kv_len + 15) // 16
    bh = np.arange(B * Hq, dtype=np.uint64)[:, None, None]
    qs = np.arange(q_start, q_start + q_len, dtype=np.uint64)[None, :, None]
    gs = np.arange(g0, g1, dtype=np.uint64)[None, None, :]
    shape = (B * Hq, q_len, g1 - g0)
    ctr = np.stack([np.broadcast_to(gs, shape), np.broadcast_to(qs, shape), np.broadcast_to(bh, shape),
                    np.full(shape, (offset // 4) & 0xFFFFFFFF, dtype=np.uint64)], -1)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint64)
    words = philox4x32_10(ctr, key).astype("<u4")
    byts = words.view(np.uint8).reshape(B * Hq, q_len, (g1 - g0) * 16)
    lo = kv_start - g0 * 16
    keep = byts[:, :, lo : lo + kv_len] >= t
    return torch.from_numpy(np.ascontiguousarray(keep)).reshape(B, Hq, q_len, kv_len)


def attention_ref_grouped_dropout(q, k, v, dout, prefix_len, keep: Tensor, p: float, doc_ids=None, scale=None):
    """R.attention_ref_grouped's fp64 math with the keep mask keep (bool [B, Hq, S, S]) and the scale s of the drop rate
    p: O = (P o Z s) V, dV = (P o Z s)^T dO, dS = P o (Z s o dP - delta), delta = rowsum(O o dO); the LSE stays that of
    the undropped P. Returns fp64 (o, lse, dq, dk, dv) like R.attention_ref_grouped."""
    B, Hq, S, D = q.shape
    Hkv = k.shape[1]
    G = Hq // Hkv
    scale = D ** -0.5 if scale is None else float(scale)
    dev, f64 = q.device, torch.float64
    prefix = [int(x) for x in prefix_len] if isinstance(prefix_len, (list, tuple, Tensor)) else [int(prefix_len)] * B
    drop_scale = attention_dropout_threshold(p)[1]
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
            pr = torch.exp(s - m)
            l = pr.sum(-1, keepdim=True)
            pr /= l
            zs = keep[b, hs].to(dev, f64) * drop_scale
            pz = pr * zs
            og = pz @ vg
            o[b, hs], lse[b, hs] = og, (m + l.log()).squeeze(-1)
            delta = (og * dog).sum(-1, keepdim=True)
            ds = pr * (zs * (dog @ vg.T) - delta)                    # dS = P o (Z s o dP - delta), then dS * scale below
            dq[b, hs] = (ds @ kg) * scale
            dk[b, hk] = torch.einsum("gqk,gqd->kd", ds, qg) * scale
            dv[b, hk] = torch.einsum("gqk,gqd->kd", pz, dog)
    return o, lse, dq, dk, dv


def transformer_layer_ref_dropout(x: Tensor, rope: Tensor, lw: R.LayerWeights, Hq: int, Hkv: int, D: int,
                                  prefix_len: int, dynamic: bool, attn_keep: Tensor, attn_p: float) -> Tensor:
    """R.transformer_layer_ref with attention dropout: the attention probabilities are formed in fp32, multiplied by
    attn_keep (bool [B, Hq, L, L]) and the scale of the drop rate attn_p, and the output is rounded to x's dtype."""
    B, L, _ = x.shape
    h = R.rmsnorm_ref(x, lw.attention_norm)
    q = R.lora_linear_ref(h, lw, "wq", dynamic).view(B, L, Hq, D)
    k = R.lora_linear_ref(h, lw, "wk", dynamic).view(B, L, Hkv, D)
    v = R.lora_linear_ref(h, lw, "wv", dynamic).view(B, L, Hkv, D)
    q = R.apply_rope(q, rope).transpose(1, 2)
    k = R.apply_rope(k, rope).transpose(1, 2)
    v = v.transpose(1, 2)
    kf, vf = (t.float().repeat_interleave(Hq // Hkv, dim=1) for t in (k, v))
    s = (q.float() @ kf.transpose(-1, -2)) * D ** -0.5
    a = torch.softmax(s.masked_fill(~R.prefix_lm_mask(L, prefix_len).to(s.device), float("-inf")), -1)
    zs = attn_keep.to(s.device, torch.float32) * attention_dropout_threshold(attn_p)[1]
    o = ((a * zs) @ vf).to(x.dtype)
    o = o.transpose(1, 2).reshape(B, L, Hq * D)
    x = x + R.lora_linear_ref(o, lw, "wo", dynamic)
    h = R.rmsnorm_ref(x, lw.ffn_norm)
    g = R.swiglu_ref(R.lora_linear_ref(h, lw, "w1", dynamic), R.lora_linear_ref(h, lw, "w3", dynamic))
    return x + R.lora_linear_ref(g, lw, "w2", dynamic)
