"""Llama decoder — drop-in for modelling/llama.py of the reference (module / parameter names, constructor and
forward signatures kept, so reference state_dicts load unchanged), with the decoder block running on this package's
sm_100a kernels.

  LlamaConfig                      llama.py:17-29      same fields
  build_rope / apply_rope          llama.py:32-73      same table [max_seq_len, head_dim/2, 2] fp32; in-place kernel
  Attention / FeedForward          llama.py:93-152     wq wk wv wo / w1 w2 w3
  TransformerLayer                 llama.py:155-174    -> FusedDecoderBlock when the base is Int8LinearWeight
  Llama                            llama.py:177-219    embed -> layers -> norm -> output -> cross-entropy

Masking: the reference wires FlexAttention `block_mask`s and dense SDPA `mask`s (llama.py:129-137). The kernels here
implement two mask families: prefix-LM  mask(q, kv) = (kv < P) | (q >= kv)  (P = 0: causal; P an int or one value per
sequence of the batch) and packed-document causal. Pass `block_mask=PrefixLM(P)` / `DocumentCausal(doc_ids)`, or — as in
the reference — a FlexAttention BlockMask or a dense boolean `mask`: those are RECOGNISED (their dense form is compared
with the family rebuilt from the descriptor read off them, `describe_dense_mask`) and raise if they are anything else.
KV caches / `input_pos` (the inference path) are out of scope and raise.
"""

from __future__ import annotations

import math
from typing import NamedTuple

import os

import torch
import torch.nn.functional as F
from torch import Tensor, nn

from .. import ops
from .fused_block import FusedDecoderBlock, block_trainables, fused_block_supported


class LlamaConfig(NamedTuple):
    embed_dim: int
    num_layers: int
    head_dim: int
    num_heads: int
    num_kv_heads: int
    intermediate_dim: int
    max_seq_len: int = 2048
    vocab_size: int = 128_256  # Llama3
    attn_dropout: float = 0.0
    rope_base: int = 50_000
    is_llama3_1: bool = False
    activation_checkpointing: bool = False


class PrefixLM:
    """Mask descriptor: keys [0, prefix_len) are visible to every query, the rest is causal. prefix_len: an int, or an
    int tensor [B] with one prefix length per sequence of the batch (utterances of different durations)."""

    def __init__(self, prefix_len):
        self.prefix_len = prefix_len if isinstance(prefix_len, Tensor) else int(prefix_len)

    def __repr__(self):
        return f"PrefixLM(prefix_len={self.prefix_len})"


class DocumentCausal:
    """Mask descriptor for packed sequences (train_metamathqa.py:51-83): tokens attend causally within their own
    document. `doc_ids` int [B, S], non-decreasing along S (documents are contiguous)."""

    prefix_len = 0

    def __init__(self, doc_ids: Tensor):
        if doc_ids.dim() == 1:
            doc_ids = doc_ids[None]
        self.doc_ids = doc_ids
        self.doc_start, self.doc_end = ops.doc_bounds(doc_ids)

    def __repr__(self):
        return f"DocumentCausal(shape={tuple(self.doc_ids.shape)})"


def document_block_mask(doc_ids: Tensor):
    """A real FlexAttention BlockMask for the document-causal mask of the reference (train_metamathqa.py:67-71),
    tagged with the document bounds so that this package's kernels accept it too."""
    from torch.nn.attention.flex_attention import create_block_mask

    ids = doc_ids.reshape(-1)

    def mask_mod(b, h, q_idx, kv_idx):
        return (ids[q_idx] == ids[kv_idx]) & (q_idx >= kv_idx)

    bm = create_block_mask(mask_mod, None, None, ids.numel(), ids.numel(), device=ids.device)
    bm.prefix_len = 0
    bm.doc_start, bm.doc_end = ops.doc_bounds(ids[None])
    return bm


def prefix_lm_block_mask(prefix_len: int, seq_len: int, device="cuda"):
    """A real FlexAttention BlockMask for the prefix-LM mask, tagged with `.prefix_len` so that both this package
    and the reference's flex_attention branch (llama.py:129-132) accept it."""
    from torch.nn.attention.flex_attention import create_block_mask

    def mask_mod(b, h, q_idx, kv_idx):
        return (kv_idx < prefix_len) | (q_idx >= kv_idx)

    bm = create_block_mask(mask_mod, None, None, seq_len, seq_len, device=device)
    bm.prefix_len = int(prefix_len)
    return bm


def _doc_bounds_of(block_mask):
    """(doc_start, doc_end) int32 [B, S] of a document mask descriptor, or (None, None)."""
    ds = getattr(block_mask, "doc_start", None)
    return (ds, getattr(block_mask, "doc_end", None)) if ds is not None else (None, None)


class _MaskDesc:
    """What the kernels understand: a prefix length (int or [B] tensor) and optional packed-document bounds."""

    def __init__(self, prefix_len=0, doc_start=None, doc_end=None):
        self.prefix_len, self.doc_start, self.doc_end = prefix_len, doc_start, doc_end


def describe_dense_mask(m: Tensor) -> _MaskDesc:
    """Recognise a dense boolean attention mask [L, L] / [B, L, L] / [B, 1, L, L] (True = attend; what the reference hands
    to SDPA, llama.py:135-137, or what a FlexAttention mask_mod evaluates to) as a member of the two families the kernels
    implement, by CONSTRUCTION AND COMPARISON: the candidate descriptor is read off the mask (row 0 gives the prefix length,
    the first visible key of each row gives its document start), the family's mask is rebuilt from it and must equal the
    input exactly. Anything else (sliding windows, arbitrary mask_mods, head-dependent masks) raises."""
    if m.dtype is not torch.bool:
        raise NotImplementedError("llamax_b200: only boolean attention masks are recognised")
    while m.dim() > 3:
        if m.shape[1] != 1 and not bool((m[:, :1] == m).all()):
            raise NotImplementedError("llamax_b200: head-dependent attention masks are not implemented")
        m = m[:, 0]
    if m.dim() == 2:
        m = m[None]
    Bm, L, L2 = m.shape
    if L != L2:
        raise NotImplementedError("llamax_b200: attention masks must be square (training path, no KV cache)")
    idx = torch.arange(L, device=m.device)
    causal = idx[:, None] >= idx[None, :]
    # --- prefix-LM: row 0 sees exactly kv < max(P, 1)
    P = m[:, 0].sum(dim=1)                                        # [Bm]
    if bool((((idx[None, None, :] < P[:, None, None]) | causal[None]) == m).all()):
        P = torch.where(P <= 1, torch.zeros_like(P), P)           # P = 1 is plain causal
        if Bm == 1 or bool((P == P[0]).all()):
            return _MaskDesc(int(P[0]))
        return _MaskDesc(P.to(torch.int32))
    # --- packed documents (train_metamathqa.py:67-70): causal inside contiguous documents
    first = m.int().argmax(dim=2)                                 # first visible key of each query row
    doc_ids = (first[:, 1:] != first[:, :-1]).cumsum(dim=1)
    doc_ids = torch.cat([torch.zeros_like(doc_ids[:, :1]), doc_ids], dim=1)
    if bool((((doc_ids[:, :, None] == doc_ids[:, None, :]) & causal[None]) == m).all()):
        ds, de = ops.doc_bounds(doc_ids)
        return _MaskDesc(0, ds, de)
    raise NotImplementedError(
        "llamax_b200: this attention mask is neither prefix-LM ((kv < P) | (q >= kv)) nor document-causal; the sm_100a "
        "kernels implement these two families (PrefixLM(P), DocumentCausal(doc_ids))")


def describe_block_mask(block_mask) -> _MaskDesc:
    """A mask descriptor of this package, or a generic FlexAttention BlockMask (llama.py:129-132): its mask_mod is evaluated
    once on the dense index grid and recognised by describe_dense_mask; the result is cached on the object."""
    if block_mask is None:
        return _MaskDesc(0)
    p = getattr(block_mask, "prefix_len", None)
    if p is not None:
        return _MaskDesc(p, *_doc_bounds_of(block_mask))
    cached = getattr(block_mask, "_llamax_desc", None)
    if cached is not None:
        return cached
    mask_mod = getattr(block_mask, "mask_mod", None)
    if mask_mod is None:
        raise NotImplementedError("llamax_b200: block_mask must be PrefixLM / DocumentCausal or a FlexAttention BlockMask")
    from torch.nn.attention.flex_attention import create_mask

    q_len, kv_len = block_mask.seq_lengths
    nb = block_mask.kv_num_blocks.shape[0]
    dense = create_mask(mask_mod, nb, 1, q_len, kv_len, device=block_mask.kv_num_blocks.device)
    desc = describe_dense_mask(dense)
    try:
        block_mask._llamax_desc = desc
    except Exception:
        pass
    return desc


_dense_desc_cache: dict = {}


def _mask_desc(mask, block_mask, input_pos) -> _MaskDesc:
    if input_pos is not None:
        raise NotImplementedError(
            "llamax_b200: `input_pos` (KV-cache inference path, llama.py:126-127) is outside the fine-tuning hot path")
    if mask is not None:
        if block_mask is not None:
            raise ValueError("pass either mask or block_mask")
        key = (mask.data_ptr(), mask._version, tuple(mask.shape), mask.device)   # the 32 layers get the same tensor
        hit = _dense_desc_cache.get(key)
        if hit is None:
            if len(_dense_desc_cache) > 8:
                _dense_desc_cache.clear()
            hit = _dense_desc_cache[key] = describe_dense_mask(mask)
        return hit
    return describe_block_mask(block_mask)


def _prefix_len_of(mask, block_mask, input_pos):
    return _mask_desc(mask, block_mask, input_pos).prefix_len


def scale_llama3_1_rope(freqs: Tensor) -> Tensor:
    """Llama-3.1 long-context frequency rescale (llama.py:32-51), vectorised."""
    factor, low, high, old_ctx = 8.0, 1.0, 4.0, 8192.0
    wavelen = 2 * torch.pi / freqs
    smooth = (old_ctx / wavelen - low) / (high - low)
    mid = (1 - smooth) * freqs / factor + smooth * freqs
    out = torch.where(wavelen < old_ctx / high, freqs, torch.where(wavelen > old_ctx / low, freqs / factor, mid))
    return out.to(freqs.dtype)


def build_rope(config: LlamaConfig) -> Tensor:
    theta = 1.0 / (config.rope_base ** (torch.arange(0, config.head_dim, 2, dtype=torch.float32) / config.head_dim))
    if config.is_llama3_1:
        theta = scale_llama3_1_rope(theta)
    angles = torch.outer(torch.arange(config.max_seq_len, dtype=torch.float32), theta)
    return torch.stack([angles.cos(), angles.sin()], dim=-1)


class _RopeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, rope: Tensor):
        B, S, H, D = x.shape
        y = x.reshape(B * S, H * D).clone()
        ops.rope_(y, rope, B, S, H, D)
        ctx.save_for_backward(rope)
        return y.view(B, S, H, D)

    @staticmethod
    def backward(ctx, dy: Tensor):
        (rope,) = ctx.saved_tensors
        B, S, H, D = dy.shape
        dx = dy.reshape(B * S, H * D).clone()
        ops.rope_(dx, rope, B, S, H, D, inverse=True)
        return dx.view(B, S, H, D), None


def apply_rope(x: Tensor, rope: Tensor) -> Tensor:
    """x [B, S, H, D]; interleaved-pair rotation in fp32 (llama.py:63-73)."""
    return _RopeFn.apply(x, rope.contiguous())


class _PrefixLMAttentionFn(torch.autograd.Function):
    """o = dropout(softmax(q k^T / sqrt(D) + mask)) v on [B, S, H, D] tensors (GQA native)."""

    @staticmethod
    def forward(ctx, q: Tensor, k: Tensor, v: Tensor, prefix_len: int, doc_start=None, doc_end=None,
                dropout_p: float = 0.0):
        B, S, Hq, D = q.shape
        Hkv = k.shape[2]
        q2, k2, v2 = (t.reshape(B * S, -1) for t in (q, k, v))
        q2, k2, v2 = (t if t.stride(1) == 1 else t.contiguous() for t in (q2, k2, v2))
        rng = ops.attn_dropout_rng(q.device) if dropout_p > 0 else None
        o, lse = ops.attn_fwd(q2, k2, v2, B, S, Hq, Hkv, D, prefix_len, doc_start=doc_start, dropout_p=dropout_p,
                              rng=rng)
        ctx.save_for_backward(q2, k2, v2, o, lse)
        ctx.dims = (B, S, Hq, Hkv, D, prefix_len)
        ctx.docs = (doc_start, doc_end)
        ctx.dropout = (dropout_p, rng)
        return o.view(B, S, Hq, D)

    @staticmethod
    def backward(ctx, do: Tensor):
        q2, k2, v2, o, lse = ctx.saved_tensors
        B, S, Hq, Hkv, D, prefix_len = ctx.dims
        dq, dk, dv = torch.empty_like(q2), torch.empty_like(k2), torch.empty_like(v2)
        ops.attn_bwd(q2, k2, v2, o, lse, do.reshape(B * S, Hq * D), dq, dk, dv, B, S, Hq, Hkv, D, prefix_len,
                     doc_start=ctx.docs[0], doc_end=ctx.docs[1], dropout_p=ctx.dropout[0], rng=ctx.dropout[1])
        return dq.view(B, S, Hq, D), dk.view(B, S, Hkv, D), dv.view(B, S, Hkv, D), None, None, None, None


def prefix_lm_attention(q: Tensor, k: Tensor, v: Tensor, prefix_len: int = 0, doc_start=None, doc_end=None,
                        dropout_p: float = 0.0) -> Tensor:
    """dropout_p > 0: attention dropout with a keep mask drawn from the default CUDA generator (ops.attn_dropout_rng)."""
    return _PrefixLMAttentionFn.apply(q, k, v, prefix_len, doc_start, doc_end, dropout_p)


class Attention(nn.Module):
    def __init__(self, config: LlamaConfig) -> None:
        super().__init__()
        self.num_heads = config.num_heads
        self.num_kv_heads = config.num_kv_heads
        self.embed_dim = config.embed_dim
        self.attn_dropout = config.attn_dropout
        self.head_dim = config.head_dim
        self.wq = nn.Linear(self.embed_dim, self.num_heads * self.head_dim, bias=False)
        self.wk = nn.Linear(self.embed_dim, self.num_kv_heads * self.head_dim, bias=False)
        self.wv = nn.Linear(self.embed_dim, self.num_kv_heads * self.head_dim, bias=False)
        self.wo = nn.Linear(self.num_heads * self.head_dim, self.embed_dim, bias=False)
        self.kv_cache = None

    def forward(self, x: Tensor, rope: Tensor, *, mask: Tensor | None = None, input_pos: Tensor | None = None,
                block_mask=None) -> Tensor:
        if self.kv_cache is not None:
            raise NotImplementedError("llamax_b200: KV-cache decoding is outside the fine-tuning hot path")
        desc = _mask_desc(mask, block_mask, input_pos)
        B, L, _ = x.shape
        q = self.wq(x).view(B, L, self.num_heads, self.head_dim)
        k = self.wk(x).view(B, L, self.num_kv_heads, self.head_dim)
        v = self.wv(x).view(B, L, self.num_kv_heads, self.head_dim)
        q, k = apply_rope(q, rope), apply_rope(k, rope)
        out = prefix_lm_attention(q, k, v, desc.prefix_len, desc.doc_start, desc.doc_end,
                                  self.attn_dropout if self.training else 0.0)
        return self.wo(out.reshape(B, L, self.num_heads * self.head_dim))


class _SwiGLUFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, ab: Tensor):
        M, F2 = ab.shape
        g, _, _ = ops.swiglu_fwd(ab[:, : F2 // 2], ab[:, F2 // 2 :])
        ctx.save_for_backward(ab)
        return g

    @staticmethod
    def backward(ctx, dg: Tensor):
        (ab,) = ctx.saved_tensors
        F_ = ab.shape[1] // 2
        dab = torch.empty_like(ab)
        ops.swiglu_bwd(dg.contiguous(), ab[:, :F_], ab[:, F_:], out_ab=dab)
        return dab


class FeedForward(nn.Module):
    def __init__(self, config: LlamaConfig):
        super().__init__()
        self.w1 = nn.Linear(config.embed_dim, config.intermediate_dim, bias=False)
        self.w3 = nn.Linear(config.embed_dim, config.intermediate_dim, bias=False)
        self.w2 = nn.Linear(config.intermediate_dim, config.embed_dim, bias=False)
        self.act = nn.SiLU()

    def forward(self, x: Tensor) -> Tensor:
        shape = x.shape
        ab = torch.cat([self.w1(x), self.w3(x)], dim=-1).reshape(-1, 2 * self.w1.out_features)
        g = _SwiGLUFn.apply(ab).view(*shape[:-1], -1)
        return self.w2(g)


class TransformerLayer(nn.Module):
    def __init__(self, config: LlamaConfig) -> None:
        super().__init__()
        self.attention_norm = nn.RMSNorm(config.embed_dim, eps=1e-5)
        self.attention = Attention(config)
        self.ffn_norm = nn.RMSNorm(config.embed_dim, eps=1e-5)
        self.feed_forward = FeedForward(config)

    def forward(self, x: Tensor, rope: Tensor, *, mask: Tensor | None = None, input_pos: Tensor | None = None,
                block_mask=None) -> Tensor:
        if fused_block_supported(self, x):
            desc = _mask_desc(mask, block_mask, input_pos)
            p = self.attention.attn_dropout if self.training else 0.0
            return FusedDecoderBlock.apply(x, rope, (self, desc.prefix_len, desc.doc_start, desc.doc_end, p),
                                           *block_trainables(self))
        # unfused composition (e.g. bf16 base weights): same math, module by module
        x = x + self.attention(self.attention_norm(x), rope, mask=mask, input_pos=input_pos, block_mask=block_mask)
        x = x + self.feed_forward(self.ffn_norm(x))
        return x


class _RMSNormFn(torch.autograd.Function):
    """nn.RMSNorm (llama.py:182, the final norm) on this package's kernels: fp32 statistics, one rounding."""

    @staticmethod
    def forward(ctx, x: Tensor, w: Tensor, eps: float):
        x2 = x.reshape(-1, x.shape[-1])
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        y, rstd, _, _ = ops.rmsnorm_fwd(x2, w.detach(), eps)
        ctx.save_for_backward(x2, w, rstd)
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy: Tensor):
        x2, w, rstd = ctx.saved_tensors
        dy2 = dy.reshape(x2.shape)
        if not dy2.is_contiguous():
            dy2 = dy2.contiguous()
        dx, dw = ops.rmsnorm_bwd(dy2, x2, w.detach(), rstd, None, want_dw=ctx.needs_input_grad[1])
        return dx.view(dy.shape), (dw.to(w.dtype) if dw is not None else None), None


def rms_norm(norm: nn.RMSNorm, x: Tensor) -> Tensor:
    w = norm.weight
    if (x.is_cuda and x.dtype is torch.bfloat16 and w is not None and w.dtype is torch.bfloat16
            and len(norm.normalized_shape) == 1 and x.shape[-1] % 8 == 0):
        return _RMSNormFn.apply(x, w, norm.eps if norm.eps is not None else torch.finfo(torch.float32).eps)
    return norm(x)


# Row compaction of the LM head (default on; LLAMAX_LM_COMPACT=0 for A/B). Positions whose label is -100 contribute
# neither to the loss nor to any gradient (F.cross_entropy(ignore_index=-100), llama.py:216-218), so the final norm,
# the [rows, vocab] logits GEMM, the cross-entropy pass and the grad_input GEMM run on the labelled rows only, gathered
# into a dense [n, D] matrix; their input gradients are scattered back into zeros. Row results of a GEMM do not depend
# on the other rows: loss and gradients are unchanged. With MetaMathQA-style batches (prompt positions masked) a
# quarter to a half of the rows drop out of the largest GEMMs of the step (vocab 128256).
# The number of labelled rows has to reach the host (GEMM sizes are host-side): it is counted by a tiny kernel at the
# START of forward() and copied to pinned memory asynchronously; by the time the host reaches the head it has queued
# the whole forward pass behind that copy, so reading the count does not drain the launch queue.
_LM_COMPACT = os.environ.get("LLAMAX_LM_COMPACT", "1") != "0"


def set_lm_compact(on: bool) -> None:
    global _LM_COMPACT
    _LM_COMPACT = bool(on)


class _LabelCount:
    """Asynchronous count of labels != -100 (one step in flight at a time; the pinned word is owned by the model)."""

    def __init__(self, owner: nn.Module, labels: Tensor):
        self.mask = labels.reshape(-1) != -100
        pin = owner.__dict__.get("_label_pin")
        if pin is None:
            pin = owner.__dict__["_label_pin"] = torch.empty(1, dtype=torch.int64, pin_memory=True)
        self.pin = pin
        pin.copy_(self.mask.sum(), non_blocking=True)
        self.event = torch.cuda.Event()
        self.event.record()

    def rows(self):
        """(n, idx): number of labelled rows and their indices in order, or (n, None) when every row is labelled."""
        self.event.synchronize()
        n = int(self.pin[0])
        if n == 0 or n == self.mask.numel():
            return n, None
        return n, torch.nonzero_static(self.mask, size=n).view(-1)


class Llama(nn.Module):
    def __init__(self, config: LlamaConfig) -> None:
        super().__init__()
        self.tok_embeddings = nn.Embedding(config.vocab_size, config.embed_dim)
        self.layers = nn.ModuleList([TransformerLayer(config) for _ in range(config.num_layers)])
        self.norm = nn.RMSNorm(config.embed_dim, eps=1e-5)
        self.output = nn.Linear(config.embed_dim, config.vocab_size, bias=False)
        self.config = config

    def build_cache(self, inference: bool = False):
        if inference:
            raise NotImplementedError("llamax_b200: build_cache(inference=True) (KV cache) is out of scope")
        device = self.tok_embeddings.weight.device
        self.register_buffer("rope", build_rope(self.config).to(device), persistent=False)

    def _run_layers(self, x: Tensor, block_mask) -> Tensor:
        rope = self.rope[: x.shape[1]]
        for layer in self.layers:
            if self.config.activation_checkpointing:
                from torch.utils.checkpoint import checkpoint

                x = checkpoint(layer, x, rope, block_mask=block_mask, use_reentrant=False)
            else:
                x = layer(x, rope, block_mask=block_mask)
        return x

    def _count_labels(self, labels: Tensor | None):
        """Called at the top of forward(): starts the asynchronous count of labelled rows (see _LM_COMPACT)."""
        if labels is None or not _LM_COMPACT or not labels.is_cuda:
            return None
        return _LabelCount(self, labels)

    def _head(self, x: Tensor, labels: Tensor | None, label_count=None) -> Tensor:
        if labels is None:
            return self.output(rms_norm(self.norm, x))
        out = self.output
        w = out.weight
        # chunked fast path only for a plain frozen-or-trainable bf16 head: `type(...) is nn.Linear` excludes LoRALinear
        # (whose adapter term the loss must see, llama.py:216 computes self.output(...)), a bias or a quantised weight
        fast = (type(out) is nn.Linear and out.bias is None and type(w) is nn.Parameter and w.is_cuda
                and w.dtype is torch.bfloat16 and x.is_cuda and x.dtype is torch.bfloat16 and w.shape[0] % 8 == 0)
        if not fast:
            logits = out(rms_norm(self.norm, x))
            return F.cross_entropy(logits.view(-1, logits.shape[-1]).float(), labels.view(-1))
        labels = labels.reshape(-1)
        x = x.reshape(-1, x.shape[-1])
        if label_count is not None:
            n, idx = label_count.rows()
            if idx is not None:   # labelled rows only, in order; index_select's backward scatters into zeros
                x = x.index_select(0, idx)
                labels = labels.index_select(0, idx)
        x = rms_norm(self.norm, x)
        return chunked_lm_loss(x, w, labels, self._output_weight_t(x))

    def _output_weight_t(self, x: Tensor):
        """W_out^T [embed, vocab] as the grad_input GEMM operand; cached while the weight is unchanged."""
        w = self.output.weight
        if not (x.requires_grad and x.is_cuda and isinstance(w, nn.Parameter) and w.dtype is torch.bfloat16):
            return None
        key = (w.data_ptr(), w._version)
        cached = getattr(self, "_w_out_t", None)
        if cached is None or cached[0] != key:
            cached = (key, w.detach().t().contiguous())
            self._w_out_t = cached
        return cached[1]

    def forward(self, x: Tensor, *, input_pos: Tensor | None = None, block_mask=None,
                labels: Tensor | None = None) -> Tensor:
        if input_pos is not None:
            raise NotImplementedError("llamax_b200: input_pos (inference) is outside the fine-tuning hot path")
        label_count = self._count_labels(labels)
        x = self.tok_embeddings(x)
        x = self._run_layers(x, block_mask)
        return self._head(x, labels, label_count)


class _ChunkedLMLoss(torch.autograd.Function):
    """mean cross-entropy of (x @ W^T).float() against labels (ignore_index = -100) without materialising the
    [M, vocab] fp32 logits (llama.py:216-218 keeps 8.4 GB of them at M = 16384). Row chunks; per chunk: bf16 logits
    by the tcgen05 bf16 GEMM, one fused cross-entropy pass that turns the logits into d(loss)/d(logits) in place,
    and dx = dlogits @ W on the same GEMM kernel (W^T is cached while the head is frozen)."""

    # rows per chunk: 8192 x 128256 bf16 logits = 2.1 GB of scratch; the dx GEMM [chunk, embed] then has 512 output
    # tiles = 6.9 waves of 74 CTA pairs (4096 rows: 3.46 waves, 13 % of the last wave idle)
    CHUNK = 8192

    @staticmethod
    def forward(ctx, x: Tensor, weight: Tensor, labels: Tensor, weight_t: Tensor | None):
        x2 = x.reshape(-1, x.shape[-1])
        if x2.stride(1) != 1:
            x2 = x2.contiguous()
        lab = labels.reshape(-1).contiguous()
        need_dx, need_dw = x.requires_grad, weight.requires_grad
        n_valid = (lab != -100).sum().clamp(min=1).float()
        inv_n = n_valid.reciprocal()
        loss_sum = torch.zeros((), device=x.device, dtype=torch.float32)
        dx = torch.empty_like(x2) if need_dx else None
        dw = torch.zeros_like(weight, dtype=torch.float32) if need_dw else None
        wd = weight.detach()
        if need_dx and weight_t is None:
            weight_t = wd.t().contiguous()
        C = _ChunkedLMLoss.CHUNK
        buf = torch.empty(min(C, x2.shape[0]), wd.shape[0], device=x.device, dtype=torch.bfloat16)
        for i in range(0, x2.shape[0], C):
            xs, ls = x2[i : i + C], lab[i : i + C]
            logits = ops.bf16_gemm(xs, wd, out=buf[: xs.shape[0]])
            ops.cross_entropy_(logits, ls, loss_sum, inv_n, need_dx or need_dw)
            if need_dx:
                ops.bf16_gemm(logits, weight_t, out=dx[i : i + C])
            if need_dw:
                dw += ops.bf16_gemm_tn(logits, xs)  # trainable head: dW chunk = dlogits^T x, operands as stored
        ctx.save_for_backward(dx, dw)
        ctx.x_shape = x.shape
        ctx.w_dtype = weight.dtype
        return loss_sum * inv_n

    @staticmethod
    def backward(ctx, g: Tensor):
        dx, dw = ctx.saved_tensors
        gx = (dx * g).view(ctx.x_shape) if dx is not None else None
        gw = (dw * g).to(ctx.w_dtype) if dw is not None else None
        return gx, gw, None, None


def chunked_lm_loss(x: Tensor, weight: Tensor, labels: Tensor, weight_t: Tensor | None = None) -> Tensor:
    from ..subclasses.int8 import Int8LinearWeight

    if (isinstance(weight, Int8LinearWeight) or not x.is_cuda or x.dtype is not torch.bfloat16
            or weight.dtype is not torch.bfloat16 or weight.shape[0] % 8):
        logits = F.linear(x, weight)  # quantised / odd head: module path + library cross-entropy
        return F.cross_entropy(logits.view(-1, logits.shape[-1]).float(), labels.view(-1))
    return _ChunkedLMLoss.apply(x, weight, labels, weight_t)
