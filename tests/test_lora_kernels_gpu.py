"""LoRA kernels against an fp64 reference, element by element, at every rank, layout and split the C ABI accepts:
the skinny projection GEMM (LoRA down-projection and dh), the LoRA term of every GEMM epilogue (ranks 4..16, any h
pitch), llamax_lora_wgrad in both forms and llamax_lora_bwd_pair.

Reference and bound. The reference is evaluated in fp64 from the very bf16 / int8 operands the kernel reads, and every
element must satisfy

    |out - ref| <= 2^-8 |ref| + C_ACC * n * 2^-24 * mag

mag is the same expression with every operand replaced by its absolute value (|A| @ |B|^T + |scale| |h| @ |B_lora|^T
+ |resid|); n counts the fp32 roundings on the way to one output: the K additions of the contraction (in any order or
tree, one product takes part in at most K - 1 of them) plus the LoRA dot product (R fmaf) plus a few scalings and
additions of the epilogue (+ 4). Each fp32 operation adds at most one unit in the last place of its result, 2^-23
relative, as long as the adder may truncate (tensor-core accumulation aligns the addends to the largest exponent and
truncates what falls off): C_ACC = 2 units of 2^-24. A bf16 store adds half a bf16 ulp, 2^-9 |value|; 2^-8 |ref|
covers it with room for the fp32 error the rounded value carries. fp32 outputs (dB, lora_wgrad) have no bf16 term.
Where the kernel itself rounds an intermediate to bf16 (the weight-only mixed GEMM rounds the accumulator before its
column scale), the bound adds 2^-8 times that intermediate's magnitude.

Every output is written into a slice of a wider, pre-filled buffer (a canary frame), and nothing outside the slice may
change. Split counts and branches named in the comments are those of a 148-SM B200.
"""
import ctypes
import math

import pytest
import torch

from llamax_b200 import _lib, ops

pytestmark = pytest.mark.gpu

U = 2.0 ** -24      # fp32 unit roundoff
C_ACC = 2           # units of U per fp32 operation (truncating adder), see the module docstring
BF16_REL = 2.0 ** -8
SCALE = 1.5         # LoRA scale of the epilogue tests: not a power of two, so a dropped or doubled scale shows


# ------------------------------------------------------------------------------------------------ helpers
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _bf16(shape, g, scale=1.0):
    return (torch.randn(*shape, device="cuda", generator=g) * scale).bfloat16()


def _i8(shape, g):
    return torch.randint(-127, 128, shape, device="cuda", dtype=torch.int8, generator=g)


def assert_fp64(out, ref, mag, n, *, bf16_out, pre=None, what=""):
    """Element-wise |out - ref| <= 2^-8 |ref| (bf16 outputs) + 2^-8 pre + C_ACC n 2^-24 mag; NaN fails."""
    assert tuple(out.shape) == tuple(ref.shape), (what, out.shape, ref.shape)
    out = out.double()
    bound = C_ACC * n * U * mag
    if bf16_out:
        bound = bound + BF16_REL * ref.abs()
    if pre is not None:
        bound = bound + BF16_REL * pre
    err = (out - ref).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = tuple(bad.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the fp64 bound; first at {i}: "
                             f"out {out[i].item():.6e} ref {ref[i].item():.6e} bound {bound[i].item():.3e}")


def _framed(rows, cols, dtype, fill, r0=1, c0=8, extra=24):
    """A [rows, cols] view at (r0, c0) of a pre-filled [rows + 2 r0, cols + extra] buffer: c0 = 8 keeps a bf16 view
    16-byte aligned, cols + extra stays a multiple of 8 when cols is. Returns (frame, view, mask of the outside)."""
    frame = torch.full((rows + 2 * r0, cols + extra), fill, dtype=dtype, device="cuda")
    mask = torch.ones_like(frame, dtype=torch.bool)
    mask[r0 : r0 + rows, c0 : c0 + cols] = False
    return frame, frame[r0 : r0 + rows, c0 : c0 + cols], mask


def _assert_untouched(frame, mask, fill, what=""):
    outside = frame[mask]
    ok = outside.isnan().all() if math.isnan(fill) else (outside == fill).all()
    assert bool(ok), f"{what}: a write landed outside the output slice"


def _lora_ref(h, lb):
    h64, b64 = h.double(), lb.double()
    return SCALE * (h64 @ b64.t()), SCALE * (h64.abs() @ b64.abs().t())


def _h_misaligned(h):
    """The same values as h in the two layouts the header allows but a 16-byte load does not: row pitch R + 4, and a
    base 4 elements (8 bytes) past a 16-byte boundary. Unused elements hold NaN, so reading them shows."""
    M, R = h.shape
    pitched = torch.full((M, R + 4), float("nan"), device="cuda", dtype=torch.bfloat16)[:, :R]
    pitched.copy_(h)
    flat = torch.full((M * R + 8,), float("nan"), device="cuda", dtype=torch.bfloat16)
    shifted = flat[4 : 4 + M * R].view(M, R)
    shifted.copy_(h)
    assert pitched.stride(0) == R + 4 and shifted.data_ptr() % 16 == 8
    return {"ldh=R+4": pitched, "base+4": shifted}


# ------------------------------------------------------------------------------------------------ skinny GEMM
# llamax_bf16_gemm without an epilogue and N <= 32 runs skinny_gemm_kernel (one CTA per 128 rows); N = 40 on the same
# operands runs the tiled GEMM: both sides of the dispatch boundary. M: single row, one row short of / past one
# 128-row block, ragged, many blocks; K: one k-block, a ragged 8-column tail, long contractions.
@pytest.mark.parametrize("M,N,K", [(1, 8, 64), (127, 16, 72), (129, 24, 4104), (300, 32, 4096), (4100, 8, 14336),
                                   (4100, 32, 4104), (129, 32, 14336), (300, 16, 64), (1, 32, 4104), (4100, 24, 72),
                                   (127, 8, 4096)])
def test_skinny_gemm_matches_fp64(M, N, K):
    g = _gen(M * 31 + N * 7 + K)
    A = _bf16((M, K + 40), g)[:, :K]                      # pitched A: lda = K + 40
    B = _bf16((40, K), g)
    a64 = A.double()
    for n in (N, 40):
        Bn = B[:n]
        # a column slice of a wider buffer at a column offset of 8: the deterministic backward's dy_cat[:, c0:c0+R] form
        frame, out, mask = _framed(M, n, torch.bfloat16, 7.0, c0=16, extra=48)
        ops.bf16_gemm(A, Bn, out=out)
        _assert_untouched(frame, mask, 7.0, f"N={n}")
        b64 = Bn.double()
        assert_fp64(out, a64 @ b64.t(), a64.abs() @ b64.abs().t(), K + 4, bf16_out=True, what=f"skinny N={n}")


# ------------------------------------------------------------------------------------------------ LoRA epilogue
# Every GEMM form with a LoRA term. The first four also run on single CTAs (ops.set_gemm_cta_group(1)); rowdot and the
# mixed-input GEMMs exist for CTA pairs only.
_CG_FORMS = ("int8", "int8_resid", "bf16", "bf16_swiglu")
_PAIR_FORMS = ("bf16_rowdot", "mixed_fwd", "mixed_bwd", "mixed_bwd_tail", "mixed_swiglu")
_EPI_CASES = [(f, cg) for f in _CG_FORMS for cg in (1, 2)] + [(f, 2) for f in _PAIR_FORMS]

# M = 2200 and N ~ 2300 give more tiles than clusters in either CTA-group mode (2 x 10 x 9 = 180 > 148 single CTAs,
# 9 x 10 = 90 > 74 pairs), so the next tile's epilogue operands are prefetched; ragged M, N and K tails throughout.
_M = 2200


def _epilogue_form(form, g):
    """(N, run, check) for one GEMM form. run(h, lb) -> tuple of outputs (each written inside a canary frame);
    check(outs, h, lb) compares them with fp64 (for the SwiGLU forms: with the two-launch path, whose GEMM is itself
    compared with fp64)."""
    M = _M
    if form in ("int8", "int8_resid"):
        N, K = 2320, 336
        A, W = _i8((M, K), g), _i8((N, K), g)
        sa = (torch.rand(M, device="cuda", generator=g) * 0.02 + 0.001).bfloat16()
        sw = (torch.rand(N, device="cuda", generator=g) * 0.002 + 0.0005).bfloat16()
        res = _bf16((M, N), g) if form == "int8_resid" else None   # a separate buffer: the pipelined-residual variant

        def run(h, lb):
            frame, out, mask = _framed(M, N, torch.bfloat16, 7.0)
            ops.int8_gemm_dequant(A, W, sa, sw, out=out, lora_h=h, lora_b=lb, lora_scale=SCALE, resid=res)
            _assert_untouched(frame, mask, 7.0, form)
            return (out,)

        def check(outs, h, lb):
            a64, w64 = A.double(), W.double()
            s = sa.double()[:, None] * sw.double()[None, :]
            lo, lo_mag = _lora_ref(h, lb)
            ref, mag = (a64 @ w64.t()) * s + lo, (a64.abs() @ w64.abs().t()) * s + lo_mag
            if res is not None:
                ref, mag = ref + res.double(), mag + res.double().abs()
            assert_fp64(outs[0], ref, mag, K + h.shape[1] + 4, bf16_out=True, what=form)

        return N, run, check

    if form == "bf16":
        N, K = 2320, 328
        A, B = _bf16((M, K), g), _bf16((N, K), g, 0.05)

        def run(h, lb):
            frame, out, mask = _framed(M, N, torch.bfloat16, 7.0)
            ops.bf16_gemm(A, B, out=out, lora_h=h, lora_b=lb, lora_scale=SCALE)
            _assert_untouched(frame, mask, 7.0, form)
            return (out,)

        def check(outs, h, lb):
            _check_bf16_gemm(outs[0], A, B, h, lb, form)

        return N, run, check

    if form == "bf16_rowdot":
        N, K, S = 2304, 328, 200                                   # N % 256 == 0, M % S == 0
        A, B, O = _bf16((M, K), g), _bf16((N, K), g, 0.05), _bf16((M, N), g)

        def run(h, lb):
            frame, C, mask = _framed(M, N, torch.bfloat16, 7.0)
            dot = torch.empty(M // S, N // 128, S, device="cuda", dtype=torch.float32)
            ep, keep = ops.make_epilogue(h, lb, SCALE)
            lib, st = ops._prep(A)
            ops._call(lib, "llamax_bf16_gemm_rowdot",
                      (ops._p(A), A.stride(0), ops._p(B), B.stride(0), ops._p(C), C.stride(0), M, N, K, ctypes.byref(ep),
                       ops._p(O), O.stride(0), ops._p(dot), S, st), "bf16_gemm")
            _assert_untouched(frame, mask, 7.0, form)
            return C, dot

        def check(outs, h, lb):
            C, dot = outs
            _check_bf16_gemm(C, A, B, h, lb, form)
            prod = C.double() * O.double()                         # the dot of the stored (bf16) C
            ref = prod.view(M // S, S, N // 128, 128).sum(-1).permute(0, 2, 1)
            mag = prod.abs().view(M // S, S, N // 128, 128).sum(-1).permute(0, 2, 1)
            assert_fp64(dot, ref, mag, 128 + 4, bf16_out=False, what="rowdot dot")

        return N, run, check

    if form == "mixed_fwd":
        N, K = 2320, 336
        x, W8 = _bf16((M, K), g), _i8((N, K), g)
        sw = (torch.rand(N, device="cuda", generator=g) * 0.01 + 1e-3).bfloat16()

        def run(h, lb):
            frame, out, mask = _framed(M, N, torch.bfloat16, 7.0)
            ops.bf16_int8_gemm(x, W8, sw, out=out, lora_h=h, lora_b=lb, lora_scale=SCALE)
            _assert_untouched(frame, mask, 7.0, form)
            return (out,)

        def check(outs, h, lb):
            x64, w64, s = x.double(), W8.double(), sw.double()[None, :]
            lo, lo_mag = _lora_ref(h, lb)
            acc = x64 @ w64.t()
            # the kernel rounds the accumulator to bf16 before the weight scale (int8.py:118): pre = |acc| * s
            assert_fp64(outs[0], acc * s + lo, (x64.abs() @ w64.abs().t()) * s + lo_mag, K + h.shape[1] + 4,
                        bf16_out=True, pre=acc.abs() * s, what=form)

        return N, run, check

    if form in ("mixed_bwd", "mixed_bwd_tail"):
        N, K1 = 2320, 320
        Rt = 8 if form == "mixed_bwd_tail" else 0
        K = K1 + Rt
        dy = _bf16((M, K + 8), g)[:, :K]                           # pitched, 16-byte aligned rows
        W8 = _i8((K1, N), g)
        s = (torch.rand(K1, device="cuda", generator=g) * 0.01 + 1e-3).bfloat16()
        tail = _bf16((Rt, N), g, 0.05) if Rt else None
        # the B operand the kernel builds: bf16(f32(w) * f32(k_scale)) (the product is exact in fp32), then the tail rows
        wt = torch.cat([(W8.float() * s.float()[:, None]).bfloat16()] + ([tail] if Rt else []), 0)

        def run(h, lb):
            frame, out, mask = _framed(M, N, torch.bfloat16, 7.0)
            ops.bf16_int8_gemm_bwd(dy, W8, s, tail=tail, out=out, lora_h=h, lora_b=lb, lora_scale=SCALE)
            _assert_untouched(frame, mask, 7.0, form)
            return (out,)

        def check(outs, h, lb):
            d64, w64 = dy.double(), wt.double()
            lo, lo_mag = _lora_ref(h, lb)
            assert_fp64(outs[0], d64 @ w64 + lo, d64.abs() @ w64.abs() + lo_mag, K + h.shape[1] + 4, bf16_out=True,
                        what=form)

        return N, run, check

    if form in ("bf16_swiglu", "mixed_swiglu"):
        N = F = 2320
        K = 320
        dy = _bf16((M, K), g)
        ab = _bf16((M, 2 * F), g)
        a, b = ab[:, :F], ab[:, F:]
        if form == "bf16_swiglu":
            wt = _bf16((F, K), g, 0.05)
        else:
            W8 = _i8((K, F), g)
            s = (torch.rand(K, device="cuda", generator=g) * 0.01 + 1e-3).bfloat16()
            wt = (W8.float() * s.float()[:, None]).bfloat16().t().contiguous()   # [F, K]: what the kernel expands

        def run(h, lb):
            frame, out_ab, mask = _framed(M, 2 * F, torch.bfloat16, 7.0)
            kw = dict(out_ab=out_ab, want_g=True, lora_h=h, lora_b=lb, lora_scale=SCALE)
            if form == "bf16_swiglu":
                _, _, gg = ops.bf16_gemm_swiglu_bwd(dy, wt, a, b, **kw)
            else:
                _, _, gg = ops.bf16_int8_gemm_swiglu_bwd(dy, W8, s, a, b, **kw)
            _assert_untouched(frame, mask, 7.0, form)
            return out_ab, gg

        def check(outs, h, lb):
            # dg = GEMM + LoRA term rounded to bf16, then the SwiGLU backward: the fused epilogue must equal the two
            # launches bit for bit, and the two-launch GEMM (same h, B, scale) must be within the fp64 bound
            dg = ops.bf16_gemm(dy, wt, lora_h=h, lora_b=lb, lora_scale=SCALE)
            _check_bf16_gemm(dg, dy, wt, h, lb, form + " dg")
            ref = torch.empty(M, 2 * F, device="cuda", dtype=torch.bfloat16)
            _, _, g_ref = ops.swiglu_bwd(dg, a, b, want_g=True, out_ab=ref)
            assert torch.equal(outs[0], ref) and torch.equal(outs[1], g_ref)

        return N, run, check

    raise ValueError(form)


def _check_bf16_gemm(out, A, B, h, lb, what):
    a64, b64 = A.double(), B.double()
    lo, lo_mag = _lora_ref(h, lb)
    assert_fp64(out, a64 @ b64.t() + lo, a64.abs() @ b64.abs().t() + lo_mag, A.shape[1] + h.shape[1] + 4,
                bf16_out=True, what=what)


def _outs_equal(x, y):
    return all(torch.equal(p, q) for p, q in zip(x, y))


@pytest.mark.parametrize("R", [4, 8, 12, 16])
@pytest.mark.parametrize("form,cg", _EPI_CASES)
def test_lora_epilogue_every_rank_matches_fp64(form, cg, R):
    """The epilogue is built for rank 8 or 16 and zero-pads a smaller runtime rank (gemm.cu, kRank): ranks 4 and 12 go
    through the unstaged path (B staged with its runtime row length, h read element by element) and must give the
    bits of rank 8 / 16 with h and B zero-padded, whose staged dot product runs the same fmaf sequence with exact
    zeros. Ranks 8 and 16 with an h row pitch of R + 4 or an h base 8 bytes off a 16-byte boundary must take the
    element-wise h reads (a 16-byte load there would be misaligned) and equal the call on the contiguous h."""
    ops.set_gemm_cta_group(cg)
    try:
        g = _gen(100 * (_CG_FORMS + _PAIR_FORMS).index(form) + R)
        N, run, check = _epilogue_form(form, g)
        h = _bf16((_M, R), g)
        lb = _bf16((N, R), g, 0.3)
        outs = run(h, lb)
        check(outs, h, lb)
        if R in (4, 12):
            pad = lambda t: torch.cat([t, torch.zeros(t.shape[0], 4, device="cuda", dtype=t.dtype)], 1)
            assert _outs_equal(run(pad(h), pad(lb)), outs), f"rank {R} differs from rank {R + 4} zero-padded"
        else:
            for name, hv in _h_misaligned(h).items():
                assert _outs_equal(run(hv, lb), outs), f"h layout {name} differs from the contiguous h"
    finally:
        ops.set_gemm_cta_group(2)


# ------------------------------------------------------------------------------------------------ lora_wgrad
def _wgrad_c(X, Ht, R, alpha, det):
    """llamax_lora_wgrad[_deterministic] through the C ABI with NaN in `out` (which the call must zero or overwrite)
    and in the whole workspace (of which only the first `splits` slices are written and read). out is the head of a
    longer NaN buffer whose tail must stay NaN."""
    M, P = X.shape
    lib, st = ops._prep(X)
    flat = torch.full((P * R + 64,), float("nan"), device="cuda", dtype=torch.float32)
    out = flat[: P * R].view(P, R)
    if det:
        ws = torch.full((_lib.LORA_WGRAD_MAX_SPLITS, P, R), float("nan"), device="cuda", dtype=torch.float32)
        ops._call(lib, "llamax_lora_wgrad_deterministic",
                  (ops._p(X), X.stride(0), ops._p(Ht), Ht.stride(0), ops._p(out), ops._p(ws), M, P, R, float(alpha), st),
                  "lora_wgrad_det")
    else:
        ops._call(lib, "llamax_lora_wgrad",
                  (ops._p(X), X.stride(0), ops._p(Ht), Ht.stride(0), ops._p(out), M, P, R, float(alpha), st), "lora_wgrad")
    assert bool(flat[P * R :].isnan().all()), "lora_wgrad wrote past out[P, R]"
    return out


def _wgrad_ref(X, H, alpha):
    x64, h64 = X.double(), H.double()
    return alpha * (x64.t() @ h64), abs(alpha) * (x64.abs().t() @ h64.abs())


# Token splits chosen by lora_wgrad_splits on 148 SMs: a cost search over 1..32 splits while 2 * P-tiles <= SMs
# (P <= 9472), else a plain count of ceil(SMs / P-tiles) = 2 for P = 14336. Splits are multiples of 64 tokens.
@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("M,P,R", [
    (1, 136, 13),         # cost search, single split of one token
    (63, 8, 1),           # cost search, single split; P smaller than one 128-row tile
    (64, 4096, 32),       # cost search, single split of exactly one k-block
    (65, 136, 4),         # cost search, 2 splits of 64: the last split is 1 token
    (1000, 520, 13),      # cost search, 16 splits of 64: the last split is 40 tokens
    (16384, 136, 4),      # cost search, 32 splits of 512 (the maximum)
    (16384, 4096, 13),    # cost search, 9 splits of 1856: the last split is 1536 tokens
    (1, 14336, 4),        # plain count, single split
    (1000, 14336, 32),    # plain count, 2 splits of 512: the last split is 488 tokens
    (16384, 14336, 1),    # plain count, 2 splits of 8192
])
def test_lora_wgrad_matches_fp64(M, P, R, det):
    g = _gen(M * 13 + P + R)
    alpha = 0.75
    X = _bf16((M, P + 24), g)[:, 8 : 8 + P]                  # pitched X, base 16 bytes into its row
    H = _bf16((M, R), g)
    Ht = ops.transposed_rank_buffer(R, M, "cuda")
    Ht.copy_(H.t())
    ref, mag = _wgrad_ref(X, H, alpha)
    out = _wgrad_c(X, Ht, R, alpha, det)
    assert_fp64(out, ref, mag, M + 2, bf16_out=False, what=f"lora_wgrad det={det}")
    if det:   # the same bits on every call: the splits are summed in split order
        assert torch.equal(_wgrad_c(X, Ht, R, alpha, det), out)


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("M,P,R", [
    (1000, 4096, 48),     # ranks 32 + 16 (the q | k | v group at rank 16); 4 splits of 256, the last 232 tokens
    (16384, 520, 64),     # ranks 32 + 32; 29 splits of 576, the last 256 tokens
])
def test_lora_wgrad_wide_rank_chunks_match_fp64(M, P, R, det):
    """ops.lora_wgrad splits ranks above the kernel's 32 accumulator columns into chunks of 32 rows of H^T."""
    g = _gen(M + P + R)
    alpha = -0.375
    X = _bf16((M, P + 24), g)[:, 8 : 8 + P]
    H = _bf16((M, R), g)
    ref, mag = _wgrad_ref(X, H, alpha)
    out = ops.lora_wgrad(X, H, alpha, deterministic=det)
    assert_fp64(out, ref, mag, M + 2, bf16_out=False, what=f"lora_wgrad R={R} det={det}")


# ------------------------------------------------------------------------------------------------ lora_bwd_pair
# llamax_lora_bwd_pair: with enough 128-token blocks to cover 3/4 of the SMs (M > 14080 on 148 SMs) one wave, no split
# of N, dh written by the CTA itself; else the N range is split and dh goes through fp32 partials in dh_accum.
@pytest.mark.parametrize("M,N,R", [
    (300, 264, 8),        # 3 column chunks: too few to split
    (2048, 14336, 16),    # 14 splits of 8 chunks: fp32 dh partials and the convert pass
    (1000, 4104, 24),     # 4 splits, the last one shorter; ragged N tail of 8 columns
    (16384, 4096, 8),     # one wave, no split
    (16384, 14336, 32),   # one wave, no split, the widest projection and rank
    (16383, 4096, 32),    # one wave, no split, ragged last token block
])
def test_lora_bwd_pair_matches_fp64(M, N, R):
    g = _gen(M + N + R)
    alpha = 0.625
    dY = _bf16((M, N + 16), g)[:, :N]
    Bt = _bf16((R, N), g, 0.05)
    H = _bf16((M, R), g)
    Ht = ops.transposed_rank_buffer(R, M, "cuda")
    Ht.copy_(H.t())
    nan = float("nan")
    dh_frame, dh, dh_mask = _framed(M, R, torch.bfloat16, nan)
    Mp = Ht.stride(0)
    dht_frame, dht, dht_mask = _framed(R, M, torch.bfloat16, nan, c0=0, extra=Mp - M + 8)
    dB_flat = torch.full((N * R + 64,), nan, device="cuda", dtype=torch.float32)
    dB = dB_flat[: N * R].view(N, R)
    acc = torch.full((M, R), nan, device="cuda", dtype=torch.float32)   # zeroed by the call when it splits
    lib, st = ops._prep(dY)
    ops._call(lib, "llamax_lora_bwd_pair",
              (ops._p(dY), dY.stride(0), ops._p(Bt), Bt.stride(0), ops._p(Ht), Ht.stride(0), ops._p(dh), dh.stride(0),
               ops._p(dht), dht.stride(0), ops._p(acc), ops._p(dB), M, N, R, float(alpha), st), "lora_wgrad")
    _assert_untouched(dh_frame, dh_mask, nan, "dh")
    _assert_untouched(dht_frame, dht_mask, nan, "dh^T")
    assert bool(dB_flat[N * R :].isnan().all()), "lora_bwd_pair wrote past dB[N, R]"
    d64, b64, h64 = dY.double(), Bt.double(), H.double()
    assert_fp64(dh, d64 @ b64.t(), d64.abs() @ b64.abs().t(), N + 2, bf16_out=True, what="dh")
    assert torch.equal(dht, dh.t())
    assert_fp64(dB, alpha * (d64.t() @ h64), abs(alpha) * (d64.abs().t() @ h64.abs()), M + 2, bf16_out=False, what="dB")
