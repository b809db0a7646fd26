"""Fused forward/backward of one Llama decoder block (TransformerLayer.forward, modelling/llama.py:163-174) for
frozen-INT8 base weights (+ optional LoRA adapters), as ONE autograd.Function over this package's kernels.

Why one Function instead of composing per-module autograd nodes:
  * the save-set is chosen by hand (x, xn, post-RoPE qkv, O + LSE, x_mid, w1x|w3x, LoRA h): ~108 KB / token / layer
    instead of the ~215 KB the eager reference keeps, so 16 k tokens x 32 layers fit HBM without recompute;
  * residual adds, LoRA up-projections and dequant scales ride in GEMM epilogues; row quantisation rides in the
    RMSNorm / SwiGLU passes; q|k|v and w1|w3 share one quantised activation and one backward GEMM
    (their grad_input GEMMs are concatenated along the contraction dimension together with the LoRA terms).

Data layout (M = B*S tokens):
  qkv   [M, (Hq + 2 Hkv) * D]   q | k | v column blocks, RoPE applied in place on q | k, read by the attention
                                kernels through strided TMA (no [B,H,S,D] transposes)
  ab    [M, 2F]                 w1 x | w3 x
  dqkv  [M, (Hq+2Hkv)*D + Rq+Rk+Rv]   gradient blocks followed by the LoRA dh columns (same for dab)
"""

from __future__ import annotations

import os

import torch
from torch import Tensor

from .. import ops
from ..subclasses.int8 import Int8LinearWeight

EPS = 1e-5

_scratch: dict = {}


def _pitch(width: int) -> int:
    """Row pitch (elements) for a bf16 GEMM operand of `width` columns: the next multiple of 64 elements = 128 bytes.
    The grad_input operands are [.., sum N + sum R] wide (6168, 28688 at 8B shape with rank 8): with the natural pitch
    every row starts 48 (or 32) bytes off a 128-byte line, so each 128-byte TMA box row straddles two lines and, at 48,
    five 32-byte sectors instead of four — measured in-step: 861 TFLOP/s on [16384, 4096, K=6168] against 1227 on
    K=28688 and 1145 on K=4096 (profiles/r2_bench_1gpu_start.json)."""
    return (width + 63) // 64 * 64


def _padded_empty(rows: int, width: int, device) -> Tensor:
    """[rows, width] bf16 view of a buffer whose row pitch is _pitch(width)."""
    return torch.empty(rows, _pitch(width), device=device, dtype=torch.bfloat16)[:, :width]


def _get_scratch(device, numel: int) -> Tensor:
    """One growing bf16 scratch per device for de-quantised weight operands (re-used by every layer)."""
    buf = _scratch.get(device)
    if buf is None or buf.numel() < numel:
        buf = torch.empty(numel, device=device, dtype=torch.bfloat16)
        _scratch[device] = buf
    return buf


# Resident backward operands. The grad_input GEMM consumes (scale * W)^T in bf16; the base weights are frozen, so on a
# 180 GB B200 the 2 B/parameter operand (14 GB for the 8B model) is built once per layer and kept, instead of being
# re-materialised from the int8 codes on every backward (224 de-quantisation launches, ~2 % of the step).
# "auto": keep an operand only while at least _CACHE_HEADROOM bytes stay free on the device after allocating it
# (checked at the first backward, i.e. at peak activation memory); "1": always; "0": never (shared scratch).
_CACHE_MODE = os.environ.get("LLAMAX_WEIGHT_CACHE", "auto")
_CACHE_HEADROOM = 24 << 30
# False: one lora_bwd_pair launch per adapter even where _group_mergeable allows one per input group (the tests' reference)
_LORA_GROUP_PAIR = True


# OPT-IN, NON-PARITY mode (SURVEY section 8 row f4; the reference author's TODO at subclasses/int8.py:105): grad_input =
# q_rowwise(dY * weight_scale) @ W_int8 on the int8 tensor path instead of the reference's bf16 (dY * s) @ bf16(W).
# The gradient is quantised to 8 bits per row, so results differ from the reference beyond the parity tolerance;
# default off, never used by bench.py's headline.
_INT8_GRAD = os.environ.get("LLAMAX_INT8_GRAD_INPUT", "0") == "1"
# OPT-IN: mixed-input GEMMs (SURVEY K4 / K5): the int8 weight is expanded to bf16 INSIDE the GEMM (converter warps between
# the TMA ring and the tensor core), so the weight-only forward needs no de-quantised scratch and grad_input needs no
# (scale * W)^T operand at all — wo and w2 are consumed as stored, q|k|v and w1|w3 as row-concatenated int8 copies
# (4.5 GB at 8B instead of 14.1 GB of bf16 operands). Results are bit-identical to the default path. Default off: at the
# 1 kW cap the kernel reaches 0.83-0.86 (grad_input) / 0.92-0.97 (forward) of the bf16-operand GEMM — the conversion's
# integer work costs more than the de-quantisation pass it removes (profiles/r2_mixed_gemm_perf.txt).
_MIXED = os.environ.get("LLAMAX_MIXED_GEMM", "0") == "1"
_ones: dict = {}


# "1": the attention backward's delta = rowsum(dO * O) comes out of the epilogue of the wo grad_input GEMM (which writes
# dO) instead of its own pass over O and dO. Measured, same box: attention-backward class 38.6 -> 36.7 ms/step, bf16 GEMM
# class 195.8 -> 197.3 (the K = 4096 GEMM is epilogue-bound and now reads O), step 401.8 vs 401.4 / 403.2: no gain at the
# power cap, so the separate pass stays the default.
_FUSE_DELTA = os.environ.get("LLAMAX_FUSE_DELTA", "0") == "1"


def set_fuse_delta(on: bool) -> None:
    global _FUSE_DELTA
    _FUSE_DELTA = bool(on)
# SURVEY K7 (opt-in): RoPE applied by the epilogue of the single q | k | v INT8 launch instead of the in-place pass over
# q | k (bit-identical; removes 2.0 ms/step of HBM pass and adds its arithmetic and a 64 B table read per 16 outputs to an
# epilogue that is the critical path at K = 4096: measured in DESIGN.md). head_dim 128, dynamic INT8, LoRA rank 0 or 8.
_ROPE_EPILOGUE = os.environ.get("LLAMAX_ROPE_EPILOGUE", "0") == "1"


def _qkv_mergeable(sq, sk, sv, nq: int, nk: int) -> bool:
    """One launch needs tile-aligned segment boundaries, one LoRA rank / scale for the three (or no LoRA at all) and
    the shape limits of the concatenated operand."""
    if nq % 256 or (nq + nk) % 256 or (nq + 2 * nk) % 64 or sq.K % 16:
        return False
    if not (sq.R == sk.R == sv.R and sq.R in (0, 8, 16)):
        return False
    return sq.R == 0 or (sq.lora_scale == sk.lora_scale == sv.lora_scale)


def set_mixed_gemm(on: bool) -> None:
    global _MIXED
    _MIXED = bool(on)


def _concat_int8_operand(cache: dict, key: str, specs):
    """Resident int8 [sum N, K] = [W_1; W_2; ...] (rows = the contraction index of grad_input) + concatenated scales; a
    single weight is used as stored (no copy). None when the shape does not fit the kernel (sum N % 64, K % 16)."""
    n_total = sum(s.N for s in specs)
    if n_total % 64 or specs[0].K % 16:
        return None
    if len(specs) == 1:
        return specs[0].w8, specs[0].ws.reshape(-1)
    sig = tuple((s.w8.data_ptr(), s.w8._version, s.ws.data_ptr(), s.ws._version) for s in specs)
    hit = cache.get(key)
    if hit is not None and hit[0] == sig:
        return hit[1], hit[2]
    w8cat = torch.cat([s.w8 for s in specs], 0).contiguous()
    scat = torch.cat([s.ws.reshape(-1) for s in specs]).contiguous()
    cache[key] = (sig, w8cat, scat)
    return w8cat, scat


def set_int8_grad_input(on: bool) -> None:
    global _INT8_GRAD
    _INT8_GRAD = bool(on)


def _ones_bf16(device, n: int) -> Tensor:
    t = _ones.get((device, n))
    if t is None:
        t = _ones[(device, n)] = torch.ones(n, device=device, dtype=torch.bfloat16)
    return t


def _i8_operand(cache: dict, key: str, specs):
    """Resident int8 [K, sum N] = [W_1; W_2; ...]^T and the concatenated weight scales [sum N] (built once)."""
    sig = tuple((s.w8.data_ptr(), s.w8._version, s.ws.data_ptr(), s.ws._version) for s in specs)
    hit = cache.get(key)
    if hit is not None and hit[0] == sig:
        return hit[1], hit[2]
    w8t = torch.cat([s.w8 for s in specs], 0).t().contiguous()
    scat = torch.cat([s.ws.reshape(-1) for s in specs]).contiguous()
    cache[key] = (sig, w8t, scat)
    return w8t, scat


def _grad_input_i8(dy: Tensor, w8t: Tensor, scat: Tensor, dh: Tensor | None, at: Tensor | None) -> Tensor:
    """dx = dequant(q(dy * scat) @ w8t^T) (+ dh @ at^T): int8 tensor path for the frozen part, LoRA term in the
    epilogue when its rank fits (<= 16), else as a second narrow bf16 GEMM accumulating into dx."""
    q, rs = ops.rowquant_int8_colscale(dy, scat)
    ones = _ones_bf16(dy.device, w8t.shape[0])
    if dh is None:
        return ops.int8_gemm_dequant(q, w8t, rs, ones)
    if dh.shape[1] <= 16:
        return ops.int8_gemm_dequant(q, w8t, rs, ones, lora_h=dh, lora_b=at, lora_scale=1.0)
    dx = ops.int8_gemm_dequant(q, w8t, rs, ones)
    return ops.bf16_gemm(dh, at, resid=dx, out=dx)


# Selective recompute (SURVEY section 8 row f4, first half): the FFN up-projections are the bulk of the block's
# save-set (w1x | w3x = 57 of 108 KB per token at 8B shape). With "ffn" the block keeps x_mid and the tiny LoRA h's
# and rebuilds xn2 (one RMSNorm pass) and ab (the w1 / w3 GEMMs, 28 % of the forward GEMM work) in its backward:
# 108 -> 43 KB per token per block for +14 % step time (w1 + w3 are 54 % of the forward GEMM work); the rebuilt tensors
# are bit-identical to the forward's. config.activation_checkpointing=True (torch checkpoint
# around the whole block, as in the reference, llama.py:209-212) remains the minimum-memory / full-recompute choice.
_RECOMPUTE = os.environ.get("LLAMAX_RECOMPUTE", "none")


def set_recompute(policy: str) -> None:
    global _RECOMPUTE
    assert policy in ("none", "ffn")
    _RECOMPUTE = policy


def set_weight_cache(mode: str) -> None:
    global _CACHE_MODE
    assert mode in ("auto", "0", "1")
    _CACHE_MODE = mode


def _operand(cache: dict | None, key: str, specs, rows: int, width: int, device):
    """bf16 [rows, width] buffer for the backward operand of `specs`.
    Returns (buffer, frozen_part_is_valid, resident): a resident buffer belongs to this layer alone (it can be
    filled ahead of its use); a non-resident one is the shared scratch."""
    numel = rows * _pitch(width)
    if cache is not None and _CACHE_MODE != "0":
        sig = (rows, width) + tuple((s.w8.data_ptr(), s.w8._version, s.ws.data_ptr(), s.ws._version) for s in specs)
        hit = cache.get(key)
        if hit is not None and hit[0] == sig and hit[1].device == device:
            return hit[1], True, True
        if hit is not None and hit[1].device == device and tuple(hit[1].shape) == (rows, width):
            cache[key] = (sig, hit[1])   # weights were overwritten in place: rebuild into the same buffer
            return hit[1], False, True
        ok = _CACHE_MODE == "1"
        if not ok:
            free, _ = torch.cuda.mem_get_info(device)
            ok = free - 2 * numel >= _CACHE_HEADROOM
        if ok:
            buf = _padded_empty(rows, width, device)
            cache[key] = (sig, buf)
            return buf, False, True
    return _get_scratch(device, numel)[:numel].view(rows, _pitch(width))[:, :width], False, False


class LinearSpec:
    """Raw tensors of one (LoRA)Linear with an Int8LinearWeight base."""

    __slots__ = ("w8", "ws", "dynamic", "lora_a", "lora_b", "lora_scale", "N", "K", "R")

    def __init__(self, module):
        w = module.weight
        if not isinstance(w, Int8LinearWeight):
            raise NotImplementedError("fused decoder block needs Int8LinearWeight base weights (quantize_linear_)")
        if module.bias is not None:
            raise NotImplementedError("fused decoder block: bias is not supported (Llama has none)")
        self.w8, self.ws, self.dynamic = w.int_data, w.scale, w.dynamic_int8_act
        self.N, self.K = w.shape
        rank = getattr(module, "rank", 0)
        if rank and rank > 0:
            self.lora_a, self.lora_b, self.lora_scale, self.R = module.lora_a, module.lora_b, float(module.scale), rank
        else:
            self.lora_a = self.lora_b = None
            self.lora_scale, self.R = 1.0, 0


def _lora_down(x: Tensor, specs) -> Tensor | None:
    """h = x @ [A_1; A_2; ...]^T for the adapters that share the input x. [M, sum R]."""
    a_list = [s.lora_a for s in specs if s.R > 0]
    if not a_list:
        return None
    a_cat = a_list[0] if len(a_list) == 1 else torch.cat(a_list, 0)
    return ops.bf16_gemm(x, a_cat.detach())


def _linear(spec: LinearSpec, x_bf16, x_q8, x_qs, h, out=None, resid=None):
    ep = {}
    if h is not None:
        ep.update(lora_h=h, lora_b=spec.lora_b.detach(), lora_scale=spec.lora_scale)
    if resid is not None:
        ep["resid"] = resid
    if spec.dynamic:
        return ops.int8_gemm_dequant(x_q8, spec.w8, x_qs, spec.ws, out=out, **ep)
    if _MIXED and spec.K % 16 == 0:
        return ops.bf16_int8_gemm(x_bf16, spec.w8, spec.ws, out=out, **ep)
    wd = ops.dequant_weight(spec.w8, None, transpose=False, apply_scale=False,
                            out=_get_scratch(x_bf16.device, spec.N * spec.K)[: spec.N * spec.K].view(spec.N, spec.K))
    return ops.bf16_gemm(x_bf16, wd, col_scale=spec.ws, round_before_scale=True, out=out, **ep)


class _GradSink:
    """Collects the fp32 -> parameter-dtype conversions of the LoRA gradients (dA^T [K,R] -> dA [R,K], dB [N,R]) so that
    they run as ONE batched launch at the end of the block's backward instead of 2-3 elementwise launches each."""

    def __init__(self):
        self.jobs = []

    def emit(self, src_f32: Tensor, transpose: bool, dtype) -> Tensor:
        if dtype is not torch.bfloat16:
            return (src_f32.t() if transpose else src_f32).to(dtype).contiguous()
        shape = (src_f32.shape[1], src_f32.shape[0]) if transpose else tuple(src_f32.shape)
        dst = torch.empty(shape, device=src_f32.device, dtype=torch.bfloat16)
        self.jobs.append((src_f32, dst, 1.0, transpose))
        return dst

    def flush(self):
        ops.batched_copy(self.jobs)
        self.jobs = []


def _lora_prepare(items, M: int, device, groups=()):
    """items: (spec, h [M,R] view, a_dst | None). ONE batched launch builds, per adapter,
    bt = scale * B^T [R,N] (operand of dh), A^T (into a_dst = its columns of a resident grad_input operand, else
    into a fresh [K,R] buffer) and ht = h^T [R,M] (operand of dB). Returns {id(spec): (bt, at, ht)}.
    groups: (key, specs, cache) for adapters that share an input and take one merged lora_bwd_pair launch: their bt
    are the diagonal blocks of one [sum R, sum N] operand (kept per layer in `cache`: the off-diagonal zeros are
    written once) and their ht consecutive rows of one [sum R, M] buffer; prep[("group", key)] = (bt_cat, ht_cat)."""
    prep, jobs = {}, []
    placed = {}
    for key, specs, cache in groups:
        if not _group_mergeable(specs):
            continue
        sig = tuple((s.R, s.N) for s in specs)
        r_tot, n_tot = sum(s.R for s in specs), sum(s.N for s in specs)
        ent = cache.get("bt_" + key)
        if ent is None or ent[0] != sig or ent[1].device != torch.device(device):
            ent = (sig, torch.zeros(r_tot, n_tot, device=device, dtype=torch.bfloat16))
            cache["bt_" + key] = ent
        bt_cat = ent[1]
        ht_cat = ops.transposed_rank_buffer(r_tot, M, device)
        r_off = n_off = 0
        for s in specs:
            placed[id(s)] = (bt_cat[r_off : r_off + s.R, n_off : n_off + s.N], ht_cat[r_off : r_off + s.R])
            r_off += s.R
            n_off += s.N
        prep[("group", key)] = (bt_cat, ht_cat)
    for s, h, a_dst in items:
        if s.R == 0:
            continue
        if id(s) in placed:
            bt, ht = placed[id(s)]
        else:
            bt = torch.empty(s.R, s.N, device=device, dtype=torch.bfloat16)
            ht = ops.transposed_rank_buffer(s.R, M, device)
        at = a_dst if a_dst is not None else torch.empty(s.K, s.R, device=device, dtype=torch.bfloat16)
        jobs += [(s.lora_b.detach(), bt, s.lora_scale, True), (s.lora_a.detach(), at, 1.0, True), (h, ht, 1.0, True)]
        prep[id(s)] = (bt, at, ht)
    ops.batched_copy(jobs)
    return prep


def _group_mergeable(specs) -> bool:
    """The adapters of linears that share an input (wq | wk | wv, w1 | w3) take ONE lora_bwd_pair launch over the
    concatenated gradient [M, sum N] with a block-diagonal scale * B^T [sum R, sum N]: dh of every adapter comes out of
    the same pass (the off-diagonal zeros contribute exact zeros) and each dB is its diagonal block of the [sum N, sum R]
    result — bit-identical to one launch per adapter, whose fixed cost (two memsets, prologue, pipeline fill and drain:
    ~25 us at the clocks of a power-capped step, more than the streaming time of the [M, 1024] wk / wv gradients) is
    paid once."""
    r_tot = sum(s.R for s in specs)
    return (_lora_pair() and _LORA_GROUP_PAIR and len(specs) > 1 and all(s.R > 0 for s in specs) and r_tot <= 32
            and all(s.lora_scale == specs[0].lora_scale for s in specs) and all(s.N % 8 == 0 for s in specs))


def _lora_pair() -> bool:
    """lora_bwd_pair reduces dB and dh across CTAs with fp32 atomics: under torch.use_deterministic_algorithms the
    two-pass form runs instead (the skinny dh GEMM streams each contraction in one CTA; lora_wgrad's deterministic form)."""
    return not ops.deterministic_mode()


def _lora_dh_dB(dy: Tensor, bt: Tensor, ht: Tensor, out_dh: Tensor, scale: float, out_dht: Tensor) -> Tensor:
    """out_dh = dy @ bt^T (bt already carries the LoRA scale), out_dht = out_dh^T (operand of the dA weight
    gradient), returns dB = scale * dy^T h (fp32)."""
    if _lora_pair():
        return ops.lora_bwd_pair(dy, bt, None, out_dh, scale, Ht=ht, out_dht=out_dht)
    ops.bf16_gemm(dy, bt, out=out_dh)
    out_dht.copy_(out_dh.t())
    return ops.lora_wgrad(dy, None, scale, Ht=ht)


def _fill_operand(wt: Tensor, valid: bool, specs):
    if valid:
        return
    n_off = 0
    for s in specs:
        ops.dequant_weight(s.w8, s.ws, transpose=True, apply_scale=True, out=wt[:, n_off : n_off + s.N])
        n_off += s.N


def _ffn_up(x1: Tensor, w_fn: Tensor, s1: LinearSpec, s3: LinearSpec, dynamic: bool, h_13: Tensor | None):
    """xn2 = RMSNorm(x1); ab = [w1 xn2 | w3 xn2] (+ LoRA). h_13 given (recompute in backward): its LoRA-down is
    skipped. Deterministic kernels: the recomputed tensors are bit-identical to the forward's."""
    xn2, rstd2, xq2, xs2 = ops.rmsnorm_fwd(x1, w_fn, EPS, quant=dynamic)
    if h_13 is None:
        h_13 = _lora_down(xn2, (s1, s3))
    F_ = s1.N
    ab = torch.empty(x1.shape[0], 2 * F_, device=x1.device, dtype=torch.bfloat16)
    _linear(s1, xn2, xq2, xs2, h_13[:, : s1.R] if s1.R > 0 else None, out=ab[:, :F_])
    _linear(s3, xn2, xq2, xs2, h_13[:, s1.R : s1.R + s3.R] if s3.R > 0 else None, out=ab[:, F_:])
    return xn2, rstd2, ab, h_13


def _group_backward(specs, dy_cat: Tensor, n_total: int, x_in: Tensor, wt: Tensor | None, a_placed: bool, prep, sink,
                    need_dx=True, i8=None, mixed=None, group_key=None):
    """Backward of linears that share one input. dy_cat [M, n_total + r_total]: gradient blocks already written in
    the first n_total columns (block i = specs[i].N columns); the LoRA dh columns are filled here. wt: the
    [K, n_total + r_total] grad_input operand (frozen part valid; A^T columns valid iff a_placed).
    Returns (dx [M,K], [(dA_i, dB_i) | None per spec])."""
    r_total = sum(s.R for s in specs)
    assert dy_cat.shape[1] == n_total + r_total
    n_off, r_off = 0, 0
    lora_grads = []
    dht = ops.transposed_rank_buffer(r_total, dy_cat.shape[0], dy_cat.device) if r_total > 0 else None
    merged = prep.get(("group", group_key)) if group_key is not None else None
    if merged is not None:   # one pass over [M, n_total] for all adapters of the group (see _group_mergeable)
        bt_cat, ht_cat = merged
        if not a_placed and i8 is None and mixed is None:
            for s in specs:
                wt[:, n_total + r_off : n_total + r_off + s.R].copy_(prep[id(s)][1])
                r_off += s.R
        dB_cat = ops.lora_bwd_pair(dy_cat[:, :n_total], bt_cat, None, dy_cat[:, n_total : n_total + r_total],
                                   specs[0].lora_scale, Ht=ht_cat, out_dht=dht)   # [n_total, r_total] fp32
        r_off = 0
        for s in specs:
            lora_grads.append([None, sink.emit(dB_cat[n_off : n_off + s.N, r_off : r_off + s.R], False, s.lora_b.dtype)])
            n_off += s.N
            r_off += s.R
        specs_loop = ()
    else:
        specs_loop = specs
    for s in specs_loop:
        dy_i = dy_cat[:, n_off : n_off + s.N]
        if s.R > 0:
            c0 = n_total + r_off
            bt, at, ht = prep[id(s)]
            if not a_placed and i8 is None and mixed is None:
                wt[:, c0 : c0 + s.R].copy_(at)
            # one pass over dy_i:  dh_i = scale * dy_i @ B_i -> columns [c0, c0+R) of dy_cat;  dB = scale * dy_i^T h_i
            dB = _lora_dh_dB(dy_i, bt, ht, dy_cat[:, c0 : c0 + s.R], s.lora_scale, dht[r_off : r_off + s.R])  # [N, R] fp32
            lora_grads.append([None, sink.emit(dB, False, s.lora_b.dtype)])
            r_off += s.R
        else:
            lora_grads.append(None)
        n_off += s.N
    if r_total > 0:
        dA_t = ops.lora_wgrad(x_in, None, 1.0, Ht=dht)  # [K, r_total] = x^T dh
        r_off = 0
        for s, lg in zip(specs, lora_grads):
            if lg is not None:
                lg[0] = sink.emit(dA_t[:, r_off : r_off + s.R], True, s.lora_a.dtype)
                r_off += s.R
    if not need_dx:
        return None, lora_grads
    if i8 is not None:   # opt-in int8 grad_input: (w8t, scat, at_cat [K, r_total] | None)
        dh = dy_cat[:, n_total:] if r_total > 0 else None
        return _grad_input_i8(dy_cat[:, :n_total], i8[0], i8[1], dh, i8[2]), lora_grads
    if mixed is not None:   # opt-in mixed-input GEMM: int8 rows as stored + the LoRA A rows as the bf16 tail
        tail = torch.cat([s.lora_a.detach() for s in specs if s.R > 0], 0) if r_total > 0 else None
        return ops.bf16_int8_gemm_bwd(dy_cat, mixed[0], mixed[1], tail=tail), lora_grads
    return ops.bf16_gemm(dy_cat, wt), lora_grads


def _single_backward(spec: LinearSpec, dy: Tensor, x_in: Tensor, wt: Tensor | None, prep, sink, i8=None, mixed=None,
                     rowdot_S: int = 0):
    """Backward of one linear whose incoming gradient buffer we do not own: LoRA term in the GEMM epilogue.
    rowdot_S > 0 (wo, head_dim 128, default bf16 operand path): the epilogue that writes dx = dO also returns the
    attention backward's delta[b, h, s] = sum_d dO * O (x_in is the attention output O): returns (dx, grads, delta)."""
    if rowdot_S > 0:
        kw = {}
        dA = dB = None
        if spec.R > 0:
            bt, at, ht = prep[id(spec)]
            dh = torch.empty(dy.shape[0], spec.R, device=dy.device, dtype=torch.bfloat16)
            dht = ops.transposed_rank_buffer(spec.R, dy.shape[0], dy.device)
            dB = sink.emit(_lora_dh_dB(dy, bt, ht, dh, spec.lora_scale, dht), False, spec.lora_b.dtype)
            kw = dict(lora_h=dh, lora_b=at, lora_scale=1.0)
        dx, delta = ops.bf16_gemm_rowdot(dy, wt, x_in, rowdot_S, **kw)
        if spec.R > 0:
            dA = sink.emit(ops.lora_wgrad(x_in, None, 1.0, Ht=dht), True, spec.lora_a.dtype)
        return dx, ((dA, dB) if spec.R > 0 else None), delta
    if spec.R > 0:
        bt, at, ht = prep[id(spec)]
        dh = torch.empty(dy.shape[0], spec.R, device=dy.device, dtype=torch.bfloat16)
        dht = ops.transposed_rank_buffer(spec.R, dy.shape[0], dy.device)
        dB = sink.emit(_lora_dh_dB(dy, bt, ht, dh, spec.lora_scale, dht), False, spec.lora_b.dtype)  # dh, dh^T, dB
        if i8 is not None:
            dx = _grad_input_i8(dy, i8[0], i8[1], dh, at)
        elif mixed is not None:
            dx = ops.bf16_int8_gemm_bwd(dy, mixed[0], mixed[1], lora_h=dh, lora_b=at, lora_scale=1.0)
        else:
            dx = ops.bf16_gemm(dy, wt, lora_h=dh, lora_b=at, lora_scale=1.0)
        dA = sink.emit(ops.lora_wgrad(x_in, None, 1.0, Ht=dht), True, spec.lora_a.dtype)
        return dx, (dA, dB)
    if i8 is not None:
        return _grad_input_i8(dy, i8[0], i8[1], None, None), None
    if mixed is not None:
        return ops.bf16_int8_gemm_bwd(dy, mixed[0], mixed[1]), None
    return ops.bf16_gemm(dy, wt), None


class FusedDecoderBlock(torch.autograd.Function):
    """out = TransformerLayer(x). Inputs after `meta` are the trainable tensors, in the order of
    `block_trainables(layer)`: attention_norm.weight, ffn_norm.weight, then (lora_a, lora_b) of
    wq, wk, wv, wo, w1, w3, w2 for the adapters that exist."""

    @staticmethod
    def forward(ctx, x: Tensor, rope: Tensor, meta, *trainables):
        layer, prefix_len, doc_start, doc_end, dropout_p = meta
        att, ff = layer.attention, layer.feed_forward
        B, S, Dm = x.shape
        M = B * S
        Hq, Hkv, D = att.num_heads, att.num_kv_heads, att.head_dim
        sq, sk, sv, so = (LinearSpec(m) for m in (att.wq, att.wk, att.wv, att.wo))
        s1, s3, s2 = (LinearSpec(m) for m in (ff.w1, ff.w3, ff.w2))
        w_an, w_fn = layer.attention_norm.weight.detach(), layer.ffn_norm.weight.detach()
        x2 = x.reshape(M, Dm)
        if not x2.is_contiguous():
            x2 = x2.contiguous()
        dyn_qkv, dyn_13 = sq.dynamic, s1.dynamic

        # --- attention half ---
        xn1, rstd1, xq, xs = ops.rmsnorm_fwd(x2, w_an, EPS, quant=dyn_qkv)
        h_qkv = _lora_down(xn1, (sq, sk, sv))
        nq, nk = Hq * D, Hkv * D
        qkv = torch.empty(M, nq + 2 * nk, device=x.device, dtype=torch.bfloat16)
        rope_done = False
        if dyn_qkv and _qkv_mergeable(sq, sk, sv, nq, nk):
            # ONE INT8 GEMM over the row-concatenated [Wq; Wk; Wv] (a resident 25 MB int8 copy per layer at 8B): N = 6144
            # instead of 4096 + 1024 + 1024 — the two N = 1024 launches fill 3.5 waves of 74 CTA pairs and ran at 1870 TOP/s
            # against 2370-2630 for the wide ones. The epilogue picks each column segment's own LoRA-h columns.
            cache = layer.__dict__.setdefault("_llamax_bwd_operands", {})
            w8cat, scat = _concat_int8_operand(cache, "wqkv_fwd", (sq, sk, sv))
            ep = {}
            if sq.R > 0:
                ep = dict(lora_h=h_qkv, lora_b=torch.cat([sq.lora_b.detach(), sk.lora_b.detach(), sv.lora_b.detach()], 0),
                          lora_scale=sq.lora_scale, lora_seg=(nq, nq + nk))
            if (_ROPE_EPILOGUE and D == 128 and sq.R in (0, 8) and (nq + nk) % 256 == 0 and rope.dtype is torch.float32
                    and rope.is_contiguous() and rope.shape[0] >= S and rope.data_ptr() % 32 == 0):
                ep["rope"] = (rope, S, nq + nk)
                rope_done = True
            ops.int8_gemm_dequant(xq, w8cat, xs, scat, out=qkv, **ep)
        else:
            r_off = 0
            for spec, c0, c1 in ((sq, 0, nq), (sk, nq, nq + nk), (sv, nq + nk, nq + 2 * nk)):
                h = h_qkv[:, r_off : r_off + spec.R] if spec.R > 0 else None
                r_off += spec.R
                _linear(spec, xn1, xq, xs, h, out=qkv[:, c0:c1])
        if not rope_done:
            ops.rope_(qkv, rope, B, S, Hq + Hkv, D)
        ctx.attn_rng = ops.attn_dropout_rng(x.device) if dropout_p > 0 else None
        o, lse = ops.attn_fwd(qkv[:, :nq], qkv[:, nq : nq + nk], qkv[:, nq + nk :], B, S, Hq, Hkv, D, prefix_len,
                              doc_start=doc_start, dropout_p=dropout_p, rng=ctx.attn_rng)
        oq = osc = None
        if so.dynamic:
            oq, osc = ops.rowquant_int8(o)
        h_o = _lora_down(o, (so,))
        x1 = _linear(so, o, oq, osc, h_o, resid=x2)

        # --- feed-forward half ---
        xn2, rstd2, ab, h_13 = _ffn_up(x1, w_fn, s1, s3, dyn_13, None)
        F_ = s1.N
        need_g = (s2.R > 0) or (not s2.dynamic)
        g, gq, gs = ops.swiglu_fwd(ab[:, :F_], ab[:, F_:], quant=s2.dynamic, want_g=need_g)
        h_2 = _lora_down(g, (s2,)) if s2.R > 0 else None
        out = _linear(s2, g, gq, gs, h_2, resid=x1)

        ctx.meta = meta
        ctx.shape = (B, S, Dm)
        # backward() re-reads the live parameters (LoRA A / B, norm weights, int8 codes / scales) instead of saving them:
        # remember their versions so that an in-place update between forward and backward raises, as autograd's own
        # saved-tensor check would, instead of silently mixing two parameter states
        ctx.versions = _param_versions(layer)
        ctx.recompute_ffn = _RECOMPUTE == "ffn"
        if ctx.recompute_ffn:   # xn2, rstd2 and ab are rebuilt from x1 in backward
            ctx.save_for_backward(x2, xn1, rstd1, qkv, o, lse, x1, h_qkv, h_o, h_13, h_2, rope)
        else:
            ctx.save_for_backward(x2, xn1, rstd1, qkv, o, lse, x1, xn2, rstd2, ab, h_qkv, h_o, h_13, h_2, rope)
        return out.view(B, S, Dm)

    @staticmethod
    def backward(ctx, dout: Tensor):
        layer, prefix_len, doc_start, doc_end, dropout_p = ctx.meta
        att, ff = layer.attention, layer.feed_forward
        if _param_versions(layer) != ctx.versions:
            raise RuntimeError("FusedDecoderBlock: a parameter of this block (LoRA A/B, norm weight or int8 weight) was "
                               "modified in place between forward and backward; its gradient would mix two states")
        if ctx.recompute_ffn:
            x2, xn1, rstd1, qkv, o, lse, x1, h_qkv, h_o, h_13, h_2, rope = ctx.saved_tensors
            s1_, s3_ = LinearSpec(ff.w1), LinearSpec(ff.w3)
            xn2, rstd2, ab, _ = _ffn_up(x1, layer.ffn_norm.weight.detach(), s1_, s3_, s1_.dynamic, h_13)
        else:
            x2, xn1, rstd1, qkv, o, lse, x1, xn2, rstd2, ab, h_qkv, h_o, h_13, h_2, rope = ctx.saved_tensors
        B, S, Dm = ctx.shape
        M = B * S
        Hq, Hkv, D = att.num_heads, att.num_kv_heads, att.head_dim
        sq, sk, sv, so = (LinearSpec(m) for m in (att.wq, att.wk, att.wv, att.wo))
        s1, s3, s2 = (LinearSpec(m) for m in (ff.w1, ff.w3, ff.w2))
        w_an, w_fn = layer.attention_norm.weight, layer.ffn_norm.weight
        F_ = s1.N
        dout2 = dout.reshape(M, Dm)
        if not dout2.is_contiguous():
            dout2 = dout2.contiguous()

        dev = dout.device
        nq, nk = Hq * D, Hkv * D
        rqkv, r13 = sq.R + sk.R + sv.R, s1.R + s3.R
        cache = layer.__dict__.setdefault("_llamax_bwd_operands", {})
        shapes = {"w2": ((s2,), s2.K, s2.N), "w13": ((s1, s3), s1.K, 2 * F_ + r13), "wo": ((so,), so.K, so.N),
                  "wqkv": ((sq, sk, sv), sq.K, nq + 2 * nk + rqkv)}
        # grad_input operands (scale * W)^T | A^T: resident ones are fetched (and, the first time, built) up front so
        # that the LoRA columns can be refreshed by the batched prepare below; the shared scratch is filled at its use
        held = {}
        i8 = {}
        mixed = {}
        if _MIXED and not _INT8_GRAD:   # opt-in: int8 weights consumed by the mixed-input GEMM, no bf16 operand
            for key, (specs, rows, width) in shapes.items():
                op = _concat_int8_operand(cache, key + "_mix", specs)
                if op is not None:
                    mixed[key] = op
        if _INT8_GRAD:   # opt-in, non-parity: int8 operands instead of the bf16 ones
            for key, (specs, rows, width) in shapes.items():
                w8t, scat = _i8_operand(cache, key + "_i8", specs)
                r_tot = sum(s.R for s in specs)
                at_cat = torch.empty(rows, r_tot, device=dev, dtype=torch.bfloat16) if (r_tot and len(specs) > 1) else None
                i8[key] = (w8t, scat, at_cat)
        else:
            for key, (specs, rows, width) in shapes.items():
                if key in mixed:
                    continue
                wt, valid, resident = _operand(cache, key, specs, rows, width, dev)
                if resident:
                    _fill_operand(wt, valid, specs)
                    held[key] = wt

        def operand(key):
            if _INT8_GRAD or key in mixed:
                return None, True
            if key in held:
                return held[key], True
            specs, rows, width = shapes[key]
            wt, valid, _ = _operand(cache, key, specs, rows, width, dev)
            _fill_operand(wt, valid, specs)
            return wt, False

        def a_dst(key, n_total, r_off, R):
            if _INT8_GRAD:
                return i8[key][2][:, r_off : r_off + R] if R > 0 else None
            if key in mixed:
                return None
            return held[key][:, n_total + r_off : n_total + r_off + R] if (key in held and R > 0) else None

        sink = _GradSink()
        prep = _lora_prepare((
            (sq, h_qkv[:, : sq.R] if sq.R else None, a_dst("wqkv", nq + 2 * nk, 0, sq.R)),
            (sk, h_qkv[:, sq.R : sq.R + sk.R] if sk.R else None, a_dst("wqkv", nq + 2 * nk, sq.R, sk.R)),
            (sv, h_qkv[:, sq.R + sk.R :] if sv.R else None, a_dst("wqkv", nq + 2 * nk, sq.R + sk.R, sv.R)),
            (so, h_o, None),
            (s1, h_13[:, : s1.R] if s1.R else None, a_dst("w13", 2 * F_, 0, s1.R)),
            (s3, h_13[:, s1.R :] if s3.R else None, a_dst("w13", 2 * F_, s1.R, s3.R)),
            (s2, h_2, None)), M, dev, groups=(("wqkv", (sq, sk, sv), cache), ("w13", (s1, s3), cache)))

        # --- w2 ---  (needs g = silu(a) * b only for dA of w2: re-materialised by the SwiGLU backward kernel)
        dab = _padded_empty(M, 2 * F_ + r13, dev)
        wt2, _ = operand("w2")
        g2 = None
        a_, b_ = ab[:, :F_], ab[:, F_:]
        # SwiGLU backward as the epilogue of the w2 grad_input GEMM: the [M, F] gradient dg never exists in HBM
        fuse = not _INT8_GRAD and F_ % 16 == 0
        dh2 = at2 = None
        if s2.R > 0:
            bt2, at2, ht2 = prep[id(s2)]
            dh2 = torch.empty(M, s2.R, device=dev, dtype=torch.bfloat16)
            dht2 = ops.transposed_rank_buffer(s2.R, M, dev)
            dB2 = sink.emit(_lora_dh_dB(dout2, bt2, ht2, dh2, s2.lora_scale, dht2), False, s2.lora_b.dtype)
        if fuse and "w2" in mixed:
            _, _, g = ops.bf16_int8_gemm_swiglu_bwd(dout2, mixed["w2"][0], mixed["w2"][1], a_, b_, out_ab=dab,
                                                    want_g=s2.R > 0, lora_h=dh2, lora_b=at2, lora_scale=1.0)
        elif fuse:   # dg = dout2 @ (s W2) (+ dh2 @ A2) goes straight through the SwiGLU backward in the GEMM epilogue
            _, _, g = ops.bf16_gemm_swiglu_bwd(dout2, wt2, a_, b_, out_ab=dab, want_g=s2.R > 0,
                                               lora_h=dh2, lora_b=at2, lora_scale=1.0)
        else:
            if _INT8_GRAD:
                dg = _grad_input_i8(dout2, i8["w2"][0], i8["w2"][1], dh2, at2)
            elif "w2" in mixed:
                dg = ops.bf16_int8_gemm_bwd(dout2, mixed["w2"][0], mixed["w2"][1], lora_h=dh2, lora_b=at2, lora_scale=1.0)
            elif s2.R > 0:
                dg = ops.bf16_gemm(dout2, wt2, lora_h=dh2, lora_b=at2, lora_scale=1.0)
            else:
                dg = ops.bf16_gemm(dout2, wt2)
            _, _, g = ops.swiglu_bwd(dg, a_, b_, want_g=s2.R > 0, out_ab=dab)
            del dg
        if s2.R > 0:
            g2 = (sink.emit(ops.lora_wgrad(g, None, 1.0, Ht=dht2), True, s2.lora_a.dtype), dB2)
        del g

        # --- w1 | w3 ---
        wt13, placed13 = operand("w13")
        dxn2, g13 = _group_backward((s1, s3), dab, 2 * F_, xn2, wt13, placed13, prep, sink, i8=i8.get("w13"),
                                    mixed=mixed.get("w13"), group_key="w13")
        del dab
        want_dw_fn, want_dw_an = w_fn.requires_grad, w_an.requires_grad
        dx1, dw_fn = ops.rmsnorm_bwd(dxn2, x1, w_fn.detach(), rstd2, dout2, want_dw=want_dw_fn)
        del dxn2

        # --- wo ---
        wto, _ = operand("wo")
        # delta = rowsum(dO * O) per head comes out of the epilogue that writes dO (no separate pass over O and dO)
        fuse_delta = (_FUSE_DELTA and wto is not None and D == 128 and (Hq * D) % 256 == 0 and not _INT8_GRAD
                      and "wo" not in mixed)
        delta = None
        if fuse_delta:
            do, go, delta = _single_backward(so, dx1, o, wto, prep, sink, rowdot_S=S)
        else:
            do, go = _single_backward(so, dx1, o, wto, prep, sink, i8=i8.get("wo"), mixed=mixed.get("wo"))

        # --- attention ---
        dqkv = _padded_empty(M, nq + 2 * nk + rqkv, dev)
        ops.attn_bwd(qkv[:, :nq], qkv[:, nq : nq + nk], qkv[:, nq + nk :], o, lse, do,
                     dqkv[:, :nq], dqkv[:, nq : nq + nk], dqkv[:, nq + nk : nq + 2 * nk], B, S, Hq, Hkv, D, prefix_len,
                     doc_start=doc_start, doc_end=doc_end, rope_inverse=rope, delta=delta,   # dq, dk come back un-rotated
                     dropout_p=dropout_p, rng=ctx.attn_rng)
        wtqkv, placedqkv = operand("wqkv")
        dxn1, gqkv = _group_backward((sq, sk, sv), dqkv, nq + 2 * nk, xn1, wtqkv, placedqkv, prep, sink,
                                     i8=i8.get("wqkv"), mixed=mixed.get("wqkv"), group_key="wqkv")
        del dqkv
        dx, dw_an = ops.rmsnorm_bwd(dxn1, x2, w_an.detach(), rstd1, dx1, want_dw=want_dw_an)
        sink.flush()   # fp32 dA^T / dB -> parameter-dtype gradients, one launch

        grads = [dw_an, dw_fn]
        for spec, g_ in zip((sq, sk, sv, so, s1, s3, s2), (*gqkv, go, *g13, g2)):
            if spec.R > 0:
                grads += [g_[0], g_[1]]
        return (dx.view(B, S, Dm), None, None, *grads)


def _param_versions(layer):
    att, ff = layer.attention, layer.feed_forward
    v = [layer.attention_norm.weight._version, layer.ffn_norm.weight._version]
    for m in (att.wq, att.wk, att.wv, att.wo, ff.w1, ff.w3, ff.w2):
        v += [m.weight.int_data._version, m.weight.scale._version]
        if getattr(m, "rank", 0) > 0:
            v += [m.lora_a._version, m.lora_b._version]
    return tuple(v)


def block_trainables(layer):
    """Tensors passed to FusedDecoderBlock.apply after `meta`, in the order backward() returns their gradients."""
    att, ff = layer.attention, layer.feed_forward
    ts = [layer.attention_norm.weight, layer.ffn_norm.weight]
    for m in (att.wq, att.wk, att.wv, att.wo, ff.w1, ff.w3, ff.w2):
        if getattr(m, "rank", 0) > 0:
            ts += [m.lora_a, m.lora_b]
    return ts


def fused_block_supported(layer, x: Tensor) -> bool:
    att, ff = layer.attention, layer.feed_forward
    mods = (att.wq, att.wk, att.wv, att.wo, ff.w1, ff.w3, ff.w2)
    return (
        x.is_cuda and x.dtype is torch.bfloat16 and att.kv_cache is None and att.head_dim in (64, 128)
        and all(isinstance(m.weight, Int8LinearWeight) and m.bias is None for m in mods)
        and all(getattr(m, "rank", 0) <= 16 and getattr(m, "rank", 0) % 8 == 0 for m in mods)
        and att.wq.weight.dynamic_int8_act == att.wk.weight.dynamic_int8_act == att.wv.weight.dynamic_int8_act
        and ff.w1.weight.dynamic_int8_act == ff.w3.weight.dynamic_int8_act
    )
