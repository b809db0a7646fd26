"""GPU parity of the tcgen05 GEMMs through the C ABI.
INT8: int32 accumulators and the dequantised bf16 output are BIT-EXACT against the oracle (subclasses/int8_mm.py).
bf16: max |err| / max |ref_fp32| <= 1e-2 (north_star tolerance)."""
import pytest
import torch

from llamax_b200 import ops
from oracle import ref_ops as R
from tests.helpers import rel_err

pytestmark = pytest.mark.gpu


def _rand_i8(*shape, gen=None):
    return torch.randint(-127, 128, shape, dtype=torch.int8, generator=gen)


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("M,N,K", [(128, 256, 128), (256, 512, 512), (300, 264, 208), (1, 8, 16), (513, 1024, 4096),
                                   (1024, 128, 1792), (77, 6144, 512)])
def test_int8_accumulators_bit_exact(cg, M, N, K):
    ops.set_gemm_cta_group(cg)
    g = torch.Generator().manual_seed(M * 7 + N)
    A, W = _rand_i8(M, K, gen=g), _rand_i8(N, K, gen=g)
    out = ops.int8_gemm_s32(A.cuda(), W.cuda()).cpu()
    assert torch.equal(out, A.int() @ W.int().T)
    ops.set_gemm_cta_group(2)


def test_int8_adversarial_range():
    """All-(+-127) operands at K = 14336: |acc| = K * 127^2 = 231,225,344 < 2^31, no saturation."""
    M, N, K = 130, 264, 14336
    A = torch.full((M, K), 127, dtype=torch.int8)
    W = torch.full((N, K), -127, dtype=torch.int8)
    W[::2] = 127
    out = ops.int8_gemm_s32(A.cuda(), W.cuda()).cpu()
    assert torch.equal(out, R.int8_mm_s32(A, W.T))
    assert out.abs().max().item() == K * 127 * 127


@pytest.mark.parametrize("M,N,K", [(512, 768, 1024), (300, 264, 208)])
def test_int8_dequant_output_bit_exact(M, N, K):
    g = torch.Generator().manual_seed(1)
    A, W = _rand_i8(M, K, gen=g), _rand_i8(N, K, gen=g)
    sa = (torch.rand(M, generator=g) * 0.1).bfloat16()
    sw = (torch.rand(N, generator=g) * 0.01).bfloat16()
    ref = R.int8_mm_dequant(A, W.T, sa, sw)
    out = ops.int8_gemm_dequant(A.cuda(), W.cuda(), sa.cuda(), sw.cuda()).cpu()
    assert torch.equal(out, ref)
    # the torch.library seam (reference schema: B is the [K,N] transposed view)
    from llamax_b200.subclasses import int8_mm_dequant

    out2 = int8_mm_dequant(A.cuda(), W.cuda().T, sa.cuda(), sw.cuda()).cpu()
    assert torch.equal(out2, ref)
    out3 = int8_mm_dequant(A.cuda(), W.T.contiguous().cuda(), sa.cuda(), sw.cuda()).cpu()  # non-view B: copied
    assert torch.equal(out3, ref)


def test_int8_full_size_checksum():
    """BASELINE config 4 at full size (M=16384, N=14336, K=4096): every row's sum of accumulators equals
    A[m,:] . colsum(W) exactly (int64) — a checksum of the whole 235 M-element result."""
    M, N, K = 16384, 14336, 4096
    g = torch.Generator(device="cuda").manual_seed(0)
    A = torch.randint(-127, 128, (M, K), dtype=torch.int8, device="cuda", generator=g)
    W = torch.randint(-127, 128, (N, K), dtype=torch.int8, device="cuda", generator=g)
    out = ops.int8_gemm_s32(A, W)
    rows = out.sum(1, dtype=torch.int64)
    wsum = W.sum(0, dtype=torch.int64).double()
    expect = (A.double() @ wsum).to(torch.int64)  # |values| < 2^53: exact in fp64
    assert torch.equal(rows, expect)
    cols = out.sum(0, dtype=torch.int64)
    expect_c = (W.double() @ A.sum(0, dtype=torch.int64).double()).to(torch.int64)
    assert torch.equal(cols, expect_c)


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (300, 264, 200), (2048, 1024, 4096), (1000, 16, 4096), (640, 4096, 6168)])
def test_bf16_gemm_tolerance(cg, M, N, K):
    ops.set_gemm_cta_group(cg)
    g = torch.Generator().manual_seed(2)
    A = torch.randn(M, K, generator=g).bfloat16()
    B = torch.randn(N, K, generator=g).bfloat16()
    out = ops.bf16_gemm(A.cuda(), B.cuda())
    assert rel_err(out, A.float() @ B.float().T) <= 1e-2
    ops.set_gemm_cta_group(2)


def test_epilogue_lora_residual_and_pitched_output():
    M, N, K, Rk = 384, 520, 512, 8
    g = torch.Generator().manual_seed(3)
    A, W = _rand_i8(M, K, gen=g), _rand_i8(N, K, gen=g)
    sa, sw = (torch.rand(M, generator=g) * 0.1).bfloat16(), (torch.rand(N, generator=g) * 0.01).bfloat16()
    h = torch.randn(M, 24, generator=g).bfloat16()            # rank-8 slice of a wider h (pitch 24)
    lb = (torch.randn(N, Rk, generator=g) * 0.1).bfloat16()
    res = torch.randn(M, N, generator=g).bfloat16()
    buf = torch.zeros(M, N + 64, dtype=torch.bfloat16, device="cuda")
    ops.int8_gemm_dequant(A.cuda(), W.cuda(), sa.cuda(), sw.cuda(), out=buf[:, 32 : 32 + N], lora_h=h.cuda()[:, 8:16],
                          lora_b=lb.cuda(), lora_scale=2.0, resid=res.cuda())
    ref = ((A.int() @ W.int().T).float() * sa.float()[:, None]) * sw.float()[None, :] \
        + 2.0 * (h[:, 8:16].float() @ lb.float().T) + res.float()
    assert rel_err(buf[:, 32 : 32 + N], ref) <= 5e-3
    assert (buf[:, :32] == 0).all() and (buf[:, 32 + N :] == 0).all()  # nothing written outside the slice


def test_weight_only_forward_and_grad_input_vs_reference_formulas():
    """int8.py:118 / :127 — bf16 reference op sequence and its fp32 evaluation."""
    M, N, K = 256, 384, 512
    g = torch.Generator().manual_seed(4)
    w8, ws = R.quantize_int8_rowwise((torch.randn(N, K, generator=g) * 0.05).bfloat16())
    x = torch.randn(M, K, generator=g).bfloat16()
    dy = torch.randn(M, N, generator=g).bfloat16()
    from llamax_b200.subclasses.int8 import int8_linear_forward, int8_linear_grad_input

    y = int8_linear_forward(x.cuda(), w8.cuda(), ws.cuda(), False).cpu()
    y_ref = R.int8_linear_fwd_ref(x, w8, ws, False)
    assert rel_err(y, R.int8_linear_fwd_f32(x, w8, ws)) <= 1e-2
    assert (y != y_ref).float().mean().item() < 0.02  # same two roundings; fp32 summation order may flip an ulp
    gx = int8_linear_grad_input(dy.cuda(), w8.cuda(), ws.cuda()).cpu()
    assert rel_err(gx, R.int8_linear_bwd_f32(dy, w8, ws)) <= 1e-2
    assert rel_err(gx, R.int8_linear_bwd_ref(dy, w8, ws).float()) <= 1e-2


def test_bad_arguments_raise():
    from llamax_b200._lib import LlamaxError

    A = torch.zeros(16, 24, dtype=torch.int8, device="cuda")  # K = 24: row pitch not 16-byte aligned
    W = torch.zeros(8, 24, dtype=torch.int8, device="cuda")
    with pytest.raises(LlamaxError):
        ops.int8_gemm_s32(A, W)
    with pytest.raises(LlamaxError):
        ops.rowquant_int8(torch.zeros(4, 16, dtype=torch.bfloat16))  # CPU tensor: no fallback


@pytest.mark.parametrize("M,N,R", [(300, 264, 8), (1024, 4096, 16), (2048, 14336, 8), (129, 128, 24), (640, 1024, 32),
                                   (16384, 4096, 8), (16384, 14336, 32), (16383, 4096, 32)])
def test_lora_bwd_pair_matches_separate_products(M, N, R):
    """Fused one-pass LoRA backward (dh = dY Bt^T and dB = alpha dY^T h) vs the fp32 products (autograd of
    modelling/lora.py:43); covers the split-N path (fp32 dh partials), the one-wave path without a split that
    M >= 111 token blocks take on 148 SMs (dh written by the CTA itself), and ragged token / column tails."""
    torch.manual_seed(M + N + R)
    dy = torch.randn(M, N + 16, device="cuda").bfloat16()[:, :N]            # pitched view
    bt = (torch.randn(R, N, device="cuda") * 0.1).bfloat16()
    h = torch.randn(M, R + 8, device="cuda").bfloat16()[:, :R]
    out = torch.zeros(M, R + 8, device="cuda", dtype=torch.bfloat16)
    dht = ops.transposed_rank_buffer(R, M, "cuda")
    dB = ops.lora_bwd_pair(dy, bt, h, out[:, :R], 0.5, out_dht=dht)
    assert torch.equal(dht, out[:, :R].t())                                   # dh^T emitted by the same pass
    dh_ref = dy.float() @ bt.float().t()
    dB_ref = 0.5 * (dy.float().t() @ h.float())
    assert rel_err(out[:, :R].float(), dh_ref) <= 1e-2
    assert rel_err(dB, dB_ref) <= 1e-2
    assert torch.count_nonzero(out[:, R:]) == 0                               # nothing written past the rank columns


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("K,M,N", [(64, 128, 256), (300, 264, 208), (1001, 512, 1536), (4096, 1024, 240), (130, 8, 8)])
def test_bf16_gemm_tn_weight_gradient_form(cg, K, M, N):
    """C = At^T Bt with both operands consumed as stored (MN-major UMMA operands), ragged K / M / N tails."""
    ops.set_gemm_cta_group(cg)
    try:
        torch.manual_seed(K + M + N)
        at = torch.randn(K, M + 8, device="cuda").bfloat16()[:, :M]      # pitched
        bt = torch.randn(K, N, device="cuda").bfloat16()
        out = ops.bf16_gemm_tn(at, bt)
        assert rel_err(out, at.float().t() @ bt.float()) <= 1e-2
    finally:
        ops.set_gemm_cta_group(2)


def test_bf16_gemm_tn_overlapping_rows():
    """Bt as an im2col view with overlapping rows (row pitch 2C < row length 3C), the audio stem's dW form."""
    torch.manual_seed(0)
    C, rows = 64, 301
    y = torch.randn(2 * rows + 4, C, device="cuda").bfloat16()
    col = y.as_strided((rows, 3 * C), (2 * C, 1))
    dz = torch.randn(rows, 128, device="cuda").bfloat16()
    out = ops.bf16_gemm_tn(dz, col)
    assert rel_err(out, dz.float().t() @ col.float()) <= 1e-2


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("M,F,K,R,pad", [(256, 512, 128, 0, 0), (301, 1792, 520, 8, 16), (1000, 464, 264, 8, 8),
                                         (130, 16, 64, 16, 16), (2048, 14336, 72, 8, 16), (301, 1792, 520, 4, 16),
                                         (1000, 464, 264, 12, 8)])
def test_gemm_with_swiglu_backward_epilogue_equals_two_launches(cg, M, F, K, R, pad):
    """The w2 grad_input GEMM with the SwiGLU backward as its epilogue (dg never written) must give exactly what
    bf16_gemm -> swiglu_bwd gives: same bf16 rounding of dg, same element formulas. Ragged M, F tails inside a tile,
    32-byte (pad 0 / 16) and 16-byte (pad 8) row alignment of the output, with and without the LoRA term and g."""
    ops.set_gemm_cta_group(cg)
    try:
        torch.manual_seed(M + F + K + R)
        dy = torch.randn(M, K, device="cuda").bfloat16()
        wt = (torch.randn(F, K, device="cuda") * 0.05).bfloat16()
        ab = torch.randn(M, 2 * F, device="cuda").bfloat16()
        a, b = ab[:, :F], ab[:, F:]
        lora = {}
        if R:
            lora = dict(lora_h=torch.randn(M, R, device="cuda").bfloat16(),
                        lora_b=(torch.randn(F, R, device="cuda") * 0.1).bfloat16(), lora_scale=1.0)
        dg = ops.bf16_gemm(dy, wt, **lora)
        ref = torch.zeros(M, 2 * F + pad, device="cuda", dtype=torch.bfloat16)
        _, _, g_ref = ops.swiglu_bwd(dg, a, b, want_g=True, out_ab=ref)
        for want_g in (True, False):
            out = torch.zeros(M, 2 * F + pad, device="cuda", dtype=torch.bfloat16)
            da, db, g = ops.bf16_gemm_swiglu_bwd(dy, wt, a, b, out_ab=out, want_g=want_g, **lora)
            assert torch.equal(out, ref)                      # da | db identical, pad columns untouched
            assert (g is None) if not want_g else torch.equal(g, g_ref)
    finally:
        ops.set_gemm_cta_group(2)


@pytest.mark.parametrize("cg", [1, 2])
@pytest.mark.parametrize("M,N,K,Rk,in_place", [(300, 512, 256, 0, False), (515, 1032, 4096, 8, False),
                                               (128, 4096, 512, 16, False), (260, 520, 128, 8, True)])
def test_int8_residual_epilogue_pipelined_reads(cg, M, N, K, Rk, in_place):
    """wo / w2 forward form: dequant + LoRA + residual (llama.py:172-173). The residual is read one 16-column group
    ahead (32-byte loads when rows are 32-byte aligned, else 16-byte; half a group at an N % 16 == 8 tail); an in-place
    call (resid is out) takes the unpipelined path. fp32 reference, same tolerance as the other dequantised outputs."""
    ops.set_gemm_cta_group(cg)
    try:
        g = torch.Generator().manual_seed(M + N + K + Rk)
        A, W = _rand_i8(M, K, gen=g), _rand_i8(N, K, gen=g)
        sa, sw = (torch.rand(M, generator=g) * 0.1).bfloat16(), (torch.rand(N, generator=g) * 0.01).bfloat16()
        res = torch.randn(M, N, generator=g).bfloat16()
        kw, lora_ref = {}, 0.0
        if Rk:
            h, lb = torch.randn(M, Rk, generator=g).bfloat16(), (torch.randn(N, Rk, generator=g) * 0.1).bfloat16()
            kw = dict(lora_h=h.cuda(), lora_b=lb.cuda(), lora_scale=1.0)
            lora_ref = h.float() @ lb.float().T
        ref = ((A.int() @ W.int().T).float() * sa.float()[:, None]) * sw.float()[None, :] + lora_ref + res.float()
        r = res.cuda()
        out = ops.int8_gemm_dequant(A.cuda(), W.cuda(), sa.cuda(), sw.cuda(), resid=r, out=r if in_place else None, **kw)
        assert rel_err(out, ref) <= 5e-3
        if not in_place:
            assert torch.equal(r.cpu(), res)                   # the residual itself is untouched
    finally:
        ops.set_gemm_cta_group(2)


@pytest.mark.parametrize("M,N,K", [(1024, 256, 8192), (1100, 264, 8200), (2048, 1024, 12288), (3000, 520, 8256)])
def test_bf16_gemm_wide_tile_path(M, N, K):
    """Long contractions (K >= 8192, M >= 1024, no epilogue) run on gemm_wide_kernel: 512 x 256 outputs per CTA-pair visit,
    two accumulators sharing the B tile. Against fp32 matmul of the same bf16 operands, ragged M / N / K included, with
    padded (128-byte) and natural operand pitches; and against the 256 x 256 kernel forced by a pitched C with an epilogue
    residual of zeros (same k order -> identical bits)."""
    torch.manual_seed(M + N)
    Kp = (K + 63) // 64 * 64
    a = (torch.randn(M, Kp, device="cuda") * 0.5).bfloat16()[:, :K]
    b = (torch.randn(N, K, device="cuda") * 0.5).bfloat16()
    c = ops.bf16_gemm(a, b)
    ref = a.float() @ b.float().t()
    assert rel_err(c, ref) <= 4e-3
    # the 256 x 256 kernel (an epilogue term disables the wide path): accumulation order over k is the same
    c2 = ops.bf16_gemm(a, b, resid=torch.zeros(M, N, device="cuda", dtype=torch.bfloat16))
    assert torch.equal(c, c2)
    # rows / columns beyond the problem are never written
    out = torch.full((M + 8, N + 8), 7.0, device="cuda", dtype=torch.bfloat16)
    ops.bf16_gemm(a, b, out=out[:M, :N])
    assert torch.equal(out[:M, :N], c) and bool((out[M:] == 7).all()) and bool((out[:, N:] == 7).all())


# ------------------------------------------------------------------------------------------------
# mixed-input GEMMs (bf16 activations x int8 weight expanded in shared memory): SURVEY K4 / K5
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,N,K,Rk,resid", [(256, 256, 64, 0, False), (512, 768, 1024, 8, True), (300, 264, 208, 0, False),
                                            (1000, 1032, 4096, 16, True), (77, 6144, 512, 8, False),
                                            (4096, 4096, 448, 0, False),    # > 74 tiles: several tiles per CTA pair
                                            (512, 768, 1024, 4, True), (300, 264, 208, 12, False)])
def test_mixed_weight_only_forward_equals_dequant_then_gemm(M, N, K, Rk, resid):
    """int8.py:118: bf16(x @ bf16(W8)^T) * scale. The in-GEMM int8 -> bf16 expansion is exact, so the mixed kernel must
    reproduce dequant_weight + bf16_gemm(round_before_scale) bit for bit, and the reference formula within 1e-2."""
    g = torch.Generator().manual_seed(M + N + K)
    x = torch.randn(M, K, generator=g).bfloat16().cuda()
    W8 = torch.randint(-128, 128, (N, K), dtype=torch.int8, generator=g).cuda()
    sw = (torch.rand(N, generator=g) * 0.01 + 1e-3).bfloat16().cuda()
    kw = {}
    if Rk:
        kw.update(lora_h=torch.randn(M, Rk, generator=g).bfloat16().cuda(),
                  lora_b=(torch.randn(N, Rk, generator=g) * 0.05).bfloat16().cuda(), lora_scale=2.0)
    if resid:
        kw["resid"] = torch.randn(M, N, generator=g).bfloat16().cuda()
    canary = torch.full((M + 2, N + 16), 7.0, device="cuda", dtype=torch.bfloat16)
    out = ops.bf16_int8_gemm(x, W8, sw, out=canary[1 : M + 1, 8 : N + 8], **kw)
    ref = ops.bf16_gemm(x, ops.dequant_weight(W8, None, transpose=False, apply_scale=False), col_scale=sw,
                        round_before_scale=True, **kw)
    assert torch.equal(out, ref)
    assert (canary[0] == 7).all() and (canary[-1] == 7).all() and (canary[:, :8] == 7).all() and (canary[:, N + 8 :] == 7).all()
    if not kw:
        y = (x.cpu().float() @ W8.cpu().float().T).bfloat16() * sw.cpu()
        assert rel_err(out, y.float()) <= 1e-2


@pytest.mark.parametrize("M,N,K1,Rt,Rk", [(256, 256, 64, 0, 0), (512, 768, 1024, 24, 0), (300, 272, 192, 8, 0),
                                          (1000, 528, 4096, 0, 8), (2048, 4096, 6144, 24, 0), (130, 512, 8192, 16, 16),
                                          (300, 272, 192, 8, 4), (1000, 528, 4096, 0, 12)])
def test_mixed_grad_input_equals_dequant_then_gemm(M, N, K1, Rt, Rk):
    """int8.py:127 with the weight consumed AS STORED ([out, in] int8, rows = contraction index), the per-row scale folded
    in during the expansion, and the LoRA A rows as a bf16 tail: bit-identical to the de-quantised-operand GEMM."""
    g = torch.Generator().manual_seed(M + N + K1 + Rt)
    K = K1 + Rt
    pitch = (K + 63) // 64 * 64
    dy = torch.zeros(M, pitch).bfloat16().cuda()[:, :K]
    dy.copy_(torch.randn(M, K, generator=g).bfloat16())
    W8 = torch.randint(-128, 128, (K1, N), dtype=torch.int8, generator=g).cuda()
    s = (torch.rand(K1, generator=g) * 0.01 + 1e-3).bfloat16().cuda()
    tail = (torch.randn(Rt, N, generator=g) * 0.05).bfloat16().cuda() if Rt else None
    kw = {}
    if Rk:
        kw.update(lora_h=torch.randn(M, Rk, generator=g).bfloat16().cuda(),
                  lora_b=(torch.randn(N, Rk, generator=g) * 0.05).bfloat16().cuda(), lora_scale=1.0)
    out = ops.bf16_int8_gemm_bwd(dy, W8, s, tail=tail, **kw)
    wt = torch.zeros(N, pitch, device="cuda", dtype=torch.bfloat16)[:, :K]
    ops.dequant_weight(W8, s, transpose=True, apply_scale=True, out=wt[:, :K1])
    if Rt:
        wt[:, K1:].copy_(tail.t())
    ref = ops.bf16_gemm(dy, wt, **kw)
    assert torch.equal(out, ref)
    if not kw:
        y = dy.cpu().float() @ torch.cat([W8.cpu().float() * s.cpu().float()[:, None]] + ([tail.cpu().float()] if Rt else []))
        assert rel_err(out, y) <= 1e-2


@pytest.mark.parametrize("M,F,K,R", [(384, 512, 256, 8), (300, 1792, 512, 0), (384, 512, 256, 4), (300, 1792, 512, 12)])
def test_mixed_grad_input_with_swiglu_backward_epilogue(M, F, K, R):
    g = torch.Generator().manual_seed(5)
    dy = torch.randn(M, K, generator=g).bfloat16().cuda()
    W8 = torch.randint(-128, 128, (K, F), dtype=torch.int8, generator=g).cuda()
    s = (torch.rand(K, generator=g) * 0.01 + 1e-3).bfloat16().cuda()
    ab = torch.randn(M, 2 * F, generator=g).bfloat16().cuda()
    kw = {}
    if R:
        kw.update(lora_h=torch.randn(M, R, generator=g).bfloat16().cuda(),
                  lora_b=(torch.randn(F, R, generator=g) * 0.05).bfloat16().cuda(), lora_scale=1.0)
    o1 = torch.empty(M, 2 * F + 16, device="cuda", dtype=torch.bfloat16)
    o2 = torch.empty_like(o1)
    da, db, g1 = ops.bf16_int8_gemm_swiglu_bwd(dy, W8, s, ab[:, :F], ab[:, F:], out_ab=o1, want_g=True, **kw)
    wt = ops.dequant_weight(W8, s, transpose=True, apply_scale=True)
    da2, db2, g2 = ops.bf16_gemm_swiglu_bwd(dy, wt, ab[:, :F], ab[:, F:], out_ab=o2, want_g=True, **kw)
    assert torch.equal(da, da2) and torch.equal(db, db2) and torch.equal(g1, g2)


def test_mixed_gemm_bad_arguments_raise():
    from llamax_b200._lib import LlamaxError

    x = torch.randn(128, 96).bfloat16().cuda()
    W8 = torch.zeros(96, 256, dtype=torch.int8).cuda()
    s = torch.ones(96).bfloat16().cuda()
    with pytest.raises(LlamaxError):   # K1 must be a multiple of 64
        ops.bf16_int8_gemm_bwd(x, W8, s)


@pytest.mark.parametrize("M,K,n0,n1,N,R", [(300, 512, 256, 512, 768, 8), (2048, 4096, 4096, 5120, 6144, 8), (515, 256, 512, 768, 1280, 16),
                                           (300, 512, 256, 512, 768, 4), (515, 256, 512, 768, 1280, 12)])
def test_int8_gemm_lora_column_segments_equal_three_launches(M, K, n0, n1, N, R):
    """q | k | v in ONE launch: column segments [0, n0), [n0, n1), [n1, N) take their own R columns of the shared LoRA-h
    matrix [M, 3R] and their own rows of the concatenated B; bit-identical to three launches on the three weights.
    Ranks 4 and 12 (zero-padded to the kernel's 8 / 16) take the per-segment h offset of the unstaged path."""
    g = torch.Generator().manual_seed(N + R)
    A, W = _rand_i8(M, K, gen=g).cuda(), _rand_i8(N, K, gen=g).cuda()
    sa = (torch.rand(M, generator=g) * 0.1).bfloat16().cuda()
    sw = (torch.rand(N, generator=g) * 0.01).bfloat16().cuda()
    h = torch.randn(M, 3 * R, generator=g).bfloat16().cuda()
    B = (torch.randn(N, R, generator=g) * 0.05).bfloat16().cuda()
    out = ops.int8_gemm_dequant(A, W, sa, sw, lora_h=h, lora_b=B, lora_scale=2.0, lora_seg=(n0, n1))
    ref = torch.empty_like(out)
    for i, (c0, c1) in enumerate(((0, n0), (n0, n1), (n1, N))):
        ops.int8_gemm_dequant(A, W[c0:c1], sa, sw[c0:c1], out=ref[:, c0:c1], lora_h=h[:, i * R : (i + 1) * R],
                              lora_b=B[c0:c1].contiguous(), lora_scale=2.0)
    assert torch.equal(out, ref)


@pytest.mark.parametrize("M,S,N,K,R", [(512, 256, 512, 256, 8), (1024, 512, 4096, 4096, 8), (300, 100, 256, 192, 0),
                                       (512, 256, 512, 256, 4), (300, 100, 256, 192, 12)])
def test_bf16_gemm_rowdot_epilogue(M, S, N, K, R):
    """The grad_input GEMM of wo also returns delta[b, h, s] = sum_d dO * O (groups of 128 columns = heads): C is
    bit-identical to the plain GEMM and the dot products equal those of the stored (rounded) C in fp32."""
    g = torch.Generator().manual_seed(M + N)
    A = torch.randn(M, K, generator=g).bfloat16().cuda()
    B = (torch.randn(N, K, generator=g) * 0.05).bfloat16().cuda()
    O = torch.randn(M, N, generator=g).bfloat16().cuda()
    kw = {}
    if R:
        kw.update(lora_h=torch.randn(M, R, generator=g).bfloat16().cuda(),
                  lora_b=(torch.randn(N, R, generator=g) * 0.05).bfloat16().cuda(), lora_scale=1.0)
    C, dot = ops.bf16_gemm_rowdot(A, B, O, S, **kw)
    assert torch.equal(C, ops.bf16_gemm(A, B, **kw))
    ref = (C.float() * O.float()).view(M // S, S, N // 128, 128).sum(-1).permute(0, 2, 1)
    assert dot.shape == ref.shape
    assert rel_err(dot, ref) <= 1e-5


def test_attention_backward_with_given_delta_equals_internal():
    B, S, Hq, Hkv, D = 2, 384, 8, 2, 128
    g = torch.Generator().manual_seed(3)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, generator=g).bfloat16().cuda()
    q, k, v = qkv[:, : Hq * D], qkv[:, Hq * D : (Hq + Hkv) * D], qkv[:, (Hq + Hkv) * D :]
    o, lse = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, 100)
    do = torch.randn(B * S, Hq * D, generator=g).bfloat16().cuda()
    outs = []
    for given in (False, True):
        d = torch.zeros_like(qkv)
        delta = None
        if given:
            delta = (do.float() * o.float()).view(B, S, Hq, D).sum(-1).permute(0, 2, 1).contiguous()
        ops.attn_bwd(q, k, v, None if given else o, lse, do, d[:, : Hq * D], d[:, Hq * D : (Hq + Hkv) * D], d[:, (Hq + Hkv) * D :],
                     B, S, Hq, Hkv, D, 100, delta=delta)
        outs.append(d)
    assert rel_err(outs[1], outs[0]) <= 2e-3


@pytest.mark.parametrize("M,S,rank", [(512, 256, 8), (600, 200, 0), (2048, 2048, 8)])
def test_int8_gemm_rope_epilogue_equals_separate_pass(M, S, rank):
    """SURVEY K7: RoPE in the epilogue of the single q | k | v INT8 launch (llamax_epilogue_t.rope) gives the bits of the
    GEMM followed by llamax_rope_inplace on its q | k columns (modelling/llama.py:63-73 on the projection's bf16 output);
    the v columns are untouched. Ragged M (rows past the last full tile), positions wrapping every S rows."""
    torch.manual_seed(M + rank)
    K, Hq, Hkv, D = 512, 8, 2, 128
    nq, nk = Hq * D, Hkv * D                       # 1024 + 256 | 256: rope_cols = 1280 = 5 tiles
    N = nq + 2 * nk
    A = torch.randint(-127, 128, (M, K), dtype=torch.int8, device="cuda")
    W = torch.randint(-127, 128, (N, K), dtype=torch.int8, device="cuda")
    a_s = (torch.rand(M, device="cuda") * 0.02 + 0.001).bfloat16()
    w_s = (torch.rand(N, device="cuda") * 0.02 + 0.001).bfloat16()
    rope = R.build_rope(D, 4096, 500000, True)[:S].contiguous().cuda()
    kw = {}
    if rank:
        kw = dict(lora_h=torch.randn(M, 3 * rank, device="cuda").bfloat16(),
                  lora_b=(torch.randn(N, rank, device="cuda") * 0.1).bfloat16(), lora_scale=2.0, lora_seg=(nq, nq + nk))
    ref = ops.int8_gemm_dequant(A, W, a_s, w_s, **kw)
    v_before = ref[:, nq + nk :].clone()
    B = (M + S - 1) // S
    pad = torch.zeros(B * S, N, dtype=torch.bfloat16, device="cuda")
    pad[:M] = ref
    ops.rope_(pad, rope, B, S, Hq + Hkv, D)         # the separate in-place pass over q | k
    fused = ops.int8_gemm_dequant(A, W, a_s, w_s, rope=(rope, S, nq + nk), **kw)
    assert torch.equal(fused[:, : nq + nk], pad[:M, : nq + nk])
    assert torch.equal(fused[:, nq + nk :], v_before)
