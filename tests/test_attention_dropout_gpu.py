"""GPU: attention dropout. The keep mask read off the production kernels equals the oracle's bit for bit, the outputs and
gradients match the fp64 oracle evaluated with the same mask, and the model paths draw, replay and reproduce it."""
import pytest
import torch

from llamax_b200 import ops
from oracle import ref_ops as R
from tests import attention_dropout_ref as DR
from tests.helpers import build_tiny_llama, oracle_layer_weights, rel_err

pytestmark = pytest.mark.gpu


def _split(qkv, Hq, Hkv, Dh):
    return qkv[:, : Hq * Dh], qkv[:, Hq * Dh : (Hq + Hkv) * Dh], qkv[:, (Hq + Hkv) * Dh :]


def _onehot_rows(n_rows, D, period=128):
    """[n_rows, D] bf16: row r is the one-hot of r % period."""
    r = torch.arange(n_rows, device="cuda")
    return (r[:, None] % period == torch.arange(D, device="cuda")[None, :]).bfloat16()


# ------------------------------------------------------------------------------------------- mask identity
# q = k = 0 gives uniform probabilities over the visible keys; with V the one-hot of kv mod 128, O[q, d] is non-zero
# exactly where Z[q, kv] keeps (kv = the visible key with kv % 128 = d). With dO the one-hot of q mod 128, dV[kv, d] is
# non-zero exactly where Z[q, kv] keeps (q with q % 128 = d): dV shows Z^T. Hq = Hkv, so no head group sums over heads.
SEEDS = [(12345, 0), ((7 << 40) + 99, 4 * 13), (2**64 - 1, 4 * (2**32 + 5))]


@pytest.mark.parametrize("seed,offset", SEEDS)
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_mask_identity_persistent_forward_and_backward(seed, offset, p):
    B, H, S, D = 2, 3, 384, 128
    qkv = torch.zeros(B * S, 3 * H * D, device="cuda", dtype=torch.bfloat16)
    q, k, v = _split(qkv, H, H, D)
    keep = DR.attention_dropout_keep(seed, offset, B, H, S, p).cuda()
    dout = _onehot_rows(B * S, D).repeat(1, H)
    for j in range(S // 128):   # one kv tile at a time: V one-hot on tile j, zero elsewhere
        v.zero_()
        v.view(B, S, H, D)[:, 128 * j : 128 * (j + 1)] = _onehot_rows(128, D)[None, :, None, :]
        o, lse = ops.attn_fwd(q, k, v, B, S, H, H, D, S, dropout_p=p, rng=(seed, offset))   # prefix S: all visible
        got = o.view(B, S, H, D).transpose(1, 2) != 0                                      # [B, H, q, d]
        assert torch.equal(got, keep[:, :, :, 128 * j : 128 * (j + 1)]), f"forward, kv tile {j}"
    v.copy_(_onehot_rows(B * S, D).repeat(1, H))
    o, lse = ops.attn_fwd(q, k, v, B, S, H, H, D, S, dropout_p=p, rng=(seed, offset))
    for det in (False, True):
        dqkv = torch.zeros_like(qkv)
        dq, dk, dv = _split(dqkv, H, H, D)
        for i in range(S // 128):   # dO one-hot on query tile i only, zero elsewhere: dV[kv, d] shows Z[128 i + d, kv]
            dsel = torch.zeros_like(dout)
            dsel.view(B, S, H * D)[:, 128 * i : 128 * (i + 1)] = dout.view(B, S, H * D)[:, 128 * i : 128 * (i + 1)]
            dqkv.zero_()
            ops.attn_bwd(q, k, v, o, lse, dsel, dq, dk, dv, B, S, H, H, D, S, deterministic=det, dropout_p=p,
                         rng=(seed, offset))
            dvt = dv.view(B, S, H, D).permute(0, 2, 3, 1) != 0                              # [B, H, d, kv]
            assert torch.equal(dvt, keep[:, :, 128 * i : 128 * (i + 1), :]), f"backward det={det}, query tile {i}"


@pytest.mark.parametrize("p", [0.1, 0.5])
def test_mask_identity_packed_documents_past_2_16(p):
    """Documents of 128 positions inside S = 65536 (attn_fwd2_kernel and the document backward): query and key
    positions up to 65535 in the counter. Causal inside a document: the identity holds on the visible pairs kv <= q."""
    B, H, S, D = 1, 2, 65536, 128
    seed, offset = 0xDEADBEEFCAFEF00D, 4 * 77
    qkv = torch.zeros(B * S, 3 * H * D, device="cuda", dtype=torch.bfloat16)
    q, k, v = _split(qkv, H, H, D)
    v.copy_(_onehot_rows(B * S, D).repeat(1, H))
    doc_ids = (torch.arange(S, device="cuda") // 128)[None]
    ds, de = ops.doc_bounds(doc_ids)
    o, lse = ops.attn_fwd(q, k, v, B, S, H, H, D, 0, doc_start=ds, dropout_p=p, rng=(seed, offset))
    dout = _onehot_rows(B * S, D).repeat(1, H)
    dqkv = torch.zeros_like(qkv)
    dq, dk, dv = _split(dqkv, H, H, D)
    ops.attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, B, S, H, H, D, 0, doc_start=ds, doc_end=de, dropout_p=p,
                 rng=(seed, offset))
    o4 = o.view(B, S, H, D).transpose(1, 2) != 0                                            # [B, H, q, kv - d0]
    dv4 = dv.view(B, S, H, D).transpose(1, 2) != 0                                          # [B, H, kv, q - d0]
    causal = torch.ones(128, 128, dtype=torch.bool, device="cuda").tril()
    for d0 in (0, 128 * 7, 65536 - 1024, 65536 - 128):   # documents at the start and past 2^16 - 1024
        keep = DR.attention_dropout_keep(seed, offset, B, H, S, p, q_start=d0, q_len=128, kv_start=d0, kv_len=128).cuda()
        assert torch.equal(o4[:, :, d0 : d0 + 128], keep & causal), f"forward, document at {d0}"
        assert torch.equal(dv4[:, :, d0 : d0 + 128].transpose(-1, -2), keep & causal), f"backward, document at {d0}"


# ------------------------------------------------------------------------------------------- parity
# (B, S, Hq, Hkv, P, head_dim, document lengths)
PARITY = [
    (2, 256, 4, 1, 0, 128, None),               # causal, GQA
    (2, 512, 8, 2, 128, 128, None),             # scalar prefix
    (2, 1756, 4, 1, [1756, 1500], 128, None),   # per-sequence prefix lengths
    (1, 301, 4, 2, 70, 128, None),              # ragged S
    (1, 640, 4, 1, 0, 128, [100, 28, 300, 212]),  # packed documents
    (2, 384, 4, 2, 100, 64, None),              # head_dim 64
    (1, 512, 4, 2, 0, 64, [200, 312]),          # head_dim 64, packed documents
]


@pytest.mark.parametrize("B,S,Hq,Hkv,P,Dh,lengths", PARITY)
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_dropout_parity_vs_fp64_oracle(B, S, Hq, Hkv, P, Dh, lengths, p):
    torch.manual_seed(S + Dh)
    seed, offset = 1000 + S, 4 * (B + Hq)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * Dh, device="cuda").bfloat16()
    dout = torch.randn(B * S, Hq * Dh, device="cuda").bfloat16()
    q, k, v = _split(qkv, Hq, Hkv, Dh)
    doc_ids = ds = de = None
    if lengths is not None:
        doc_ids = torch.repeat_interleave(torch.arange(len(lengths)), torch.tensor(lengths))[None].expand(B, S).cuda()
        ds, de = ops.doc_bounds(doc_ids)
    Pd = torch.tensor(P, device="cuda", dtype=torch.int32) if isinstance(P, list) else P
    keep = DR.attention_dropout_keep(seed, offset, B, Hq, S, p).cuda()
    to4 = lambda t, H: t.reshape(B, S, H, Dh).transpose(1, 2)
    o_r, lse_r, dq_r, dk_r, dv_r = DR.attention_ref_grouped_dropout(
        to4(q, Hq), to4(k, Hkv), to4(v, Hkv), to4(dout, Hq), P, keep, p, doc_ids=doc_ids)
    o, lse = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, Dh, Pd, doc_start=ds, dropout_p=p, rng=(seed, offset))
    assert rel_err(to4(o, Hq), o_r) <= 1e-2
    assert (lse.double() - lse_r).abs().max().item() < 1e-3
    grads = {}
    for det in (False, True):
        dqkv = torch.zeros_like(qkv)
        dq, dk, dv = _split(dqkv, Hq, Hkv, Dh)
        ops.attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, B, S, Hq, Hkv, Dh, Pd, doc_start=ds, doc_end=de,
                     deterministic=det, dropout_p=p, rng=(seed, offset))
        assert rel_err(to4(dq, Hq), dq_r) <= 1e-2, f"dq det={det}"
        assert rel_err(to4(dk, Hkv), dk_r) <= 1e-2, f"dk det={det}"
        assert rel_err(to4(dv, Hkv), dv_r) <= 1e-2, f"dv det={det}"
        grads[det] = (dk.clone(), dv.clone())
    # the deterministic dK / dV come from the same MMA order: bitwise those of the default backward
    assert torch.equal(grads[True][0], grads[False][0]) and torch.equal(grads[True][1], grads[False][1])


def test_zero_p_and_eval_are_todays_kernels():
    B, S, Hq, Hkv, D = 2, 512, 8, 2, 128
    torch.manual_seed(5)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * D, device="cuda").bfloat16()
    dout = torch.randn(B * S, Hq * D, device="cuda").bfloat16()
    q, k, v = _split(qkv, Hq, Hkv, D)
    o0, l0 = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, 64)
    o1, l1 = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, 64, dropout_p=0.0)
    o2, l2 = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, 64, dropout_p=0.001, rng=(1, 0))   # round(256 p) = 0
    assert torch.equal(o0, o1) and torch.equal(o0, o2) and torch.equal(l0, l1) and torch.equal(l0, l2)
    outs = []
    for p, rng in ((0.0, None), (0.001, (1, 0))):
        g = torch.zeros_like(qkv)
        ops.attn_bwd(q, k, v, o0, l0, dout, *_split(g, Hq, Hkv, D), B, S, Hq, Hkv, D, 64, deterministic=True,
                     dropout_p=p, rng=rng)
        outs.append(g)
    assert torch.equal(outs[0], outs[1])
    with pytest.raises(ValueError):
        ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, 64, dropout_p=1.0)
    with pytest.raises(ValueError):
        ops.attn_bwd(q, k, v, o0, l0, dout, *_split(torch.zeros_like(qkv), Hq, Hkv, D), B, S, Hq, Hkv, D, 64,
                     dropout_p=0.1)   # no rng


# ------------------------------------------------------------------------------------------- model paths
def _model(p, dynamic=True, num_layers=2, ckpt=False, fused=True):
    model = build_tiny_llama(dynamic, num_layers=num_layers)
    model.config = model.config._replace(activation_checkpointing=ckpt)
    for layer in model.layers:
        layer.attention.attn_dropout = p
    model = model.cuda()
    model.build_cache()
    model.tok_embeddings.requires_grad_(False)
    model.output.requires_grad_(False)
    return model


def _step(model, tokens, labels, seed, P=40):
    from llamax_b200.modelling import PrefixLM

    for prm in model.parameters():
        prm.grad = None
    torch.manual_seed(seed)
    loss = model(tokens, labels=labels, block_mask=PrefixLM(P))
    loss.backward()
    return loss.item(), [prm.grad.clone() for prm in model.parameters() if prm.grad is not None]


def _batch():
    g = torch.Generator().manual_seed(13)
    tokens = torch.randint(0, 1024, (2, 160), generator=g).cuda()
    labels = torch.randint(0, 1024, (2, 160), generator=g).cuda()
    return tokens, labels


def test_model_masks_fresh_per_call_and_reproducible():
    tokens, labels = _batch()
    model = _model(0.1)
    l0, g0 = _step(model, tokens, labels, 7)
    l1, g1 = _step(model, tokens, labels, 7)
    l2, _ = _step(model, tokens, labels, 8)
    assert abs(l0 - l1) <= 1e-5 * abs(l0) and l0 != l2
    assert all(rel_err(a, b) <= 2e-2 for a, b in zip(g0, g1))
    # two forwards in a row draw different masks
    from llamax_b200.modelling import PrefixLM

    with torch.no_grad():
        torch.manual_seed(7)
        a = model(tokens, block_mask=PrefixLM(40))
        b = model(tokens, block_mask=PrefixLM(40))
    assert not torch.equal(a, b)
    # eval mode: no dropout, bitwise the p = 0 model
    ref = _model(0.0).eval()
    model.eval()
    with torch.no_grad():
        assert torch.equal(model(tokens, block_mask=PrefixLM(40)), ref(tokens, block_mask=PrefixLM(40)))


@pytest.mark.parametrize("det", [False, True])
def test_activation_checkpointing_replays_the_mask(det):
    tokens, labels = _batch()
    prev = torch.are_deterministic_algorithms_enabled()
    fill = torch.utils.deterministic.fill_uninitialized_memory
    try:
        torch.use_deterministic_algorithms(det)
        torch.utils.deterministic.fill_uninitialized_memory = False
        plain = _step(_model(0.1), tokens, labels, 21)
        ckpt = _step(_model(0.1, ckpt=True), tokens, labels, 21)
        if det:
            assert plain[0] == ckpt[0] and all(torch.equal(a, b) for a, b in zip(plain[1], ckpt[1]))
            again = _step(_model(0.1), tokens, labels, 21)
            assert plain[0] == again[0] and all(torch.equal(a, b) for a, b in zip(plain[1], again[1]))
        else:
            assert abs(plain[0] - ckpt[0]) <= 1e-5 * abs(plain[0])
            assert all(rel_err(a, b) <= 2e-2 for a, b in zip(plain[1], ckpt[1]))
    finally:
        torch.use_deterministic_algorithms(prev)
        torch.utils.deterministic.fill_uninitialized_memory = fill


@pytest.mark.parametrize("recompute", [False, True])
def test_fused_block_matches_oracle_with_the_same_mask(recompute, monkeypatch):
    """One block at dim 512 (GQA 4 / 1, head_dim 128), prefix 100, p = 0.1: output and input gradient against the fp32
    evaluation of the reference op sequence with the mask the block drew."""
    from llamax_b200.modelling import PrefixLM, fused_block

    monkeypatch.setattr(fused_block, "_RECOMPUTE", "ffn" if recompute else "none")
    _block_case(build_tiny_llama(True, num_layers=1), B=2, S=320, P=100, p=0.1)


def test_fused_block_8b_shape_matches_oracle_with_the_same_mask():
    from llamax_b200.modelling import LlamaConfig

    cfg = LlamaConfig(4096, 1, 128, 32, 8, 14336, max_seq_len=512, vocab_size=1024, rope_base=500000, is_llama3_1=True)
    _block_case(build_tiny_llama(True, num_layers=1, config=cfg), B=1, S=512, P=300, p=0.1)


def _block_case(model, B, S, P, p):
    from llamax_b200.modelling import PrefixLM
    from llamax_b200.modelling.fused_block import fused_block_supported

    layer = model.layers[0]
    cfg = model.config
    layer.attention.attn_dropout = p
    rope = R.build_rope(cfg.head_dim, cfg.max_seq_len, cfg.rope_base, cfg.is_llama3_1)[:S]
    torch.manual_seed(3)
    x = torch.randn(B, S, cfg.embed_dim).bfloat16()
    dout = torch.randn(B, S, cfg.embed_dim).bfloat16()
    lw = oracle_layer_weights(layer, torch.float32)
    layer = layer.cuda()
    xc = x.detach().clone().cuda().requires_grad_(True)
    assert fused_block_supported(layer, xc)
    torch.manual_seed(11)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    seed, offset = gen.initial_seed(), gen.get_offset()
    out = layer(xc, rope.cuda(), block_mask=PrefixLM(P))
    out.backward(dout.cuda())
    keep = DR.attention_dropout_keep(seed, offset, B, cfg.num_heads, S, p)
    xr = x.detach().clone().float().requires_grad_(True)
    ref = DR.transformer_layer_ref_dropout(xr, rope, lw, cfg.num_heads, cfg.num_kv_heads, cfg.head_dim, P, True, keep, p)
    ref.backward(dout.float())
    assert rel_err(out, ref) <= 1e-2 and rel_err(xc.grad, xr.grad) <= 1e-2
    assert rel_err(layer.attention.wv.lora_b.grad, lw.lora_b["wv"].grad) <= 2e-2


def test_unfused_attention_module_matches_oracle():
    """Attention.forward on bf16 weights (no fused block): prefix_lm_attention with dropout, against the oracle."""
    from llamax_b200.modelling import prefix_lm_attention

    B, S, Hq, Hkv, D, P, p = 2, 300, 4, 2, 128, 50, 0.5
    torch.manual_seed(2)
    q = torch.randn(B, S, Hq, D, device="cuda").bfloat16().requires_grad_(True)
    k = torch.randn(B, S, Hkv, D, device="cuda").bfloat16().requires_grad_(True)
    v = torch.randn(B, S, Hkv, D, device="cuda").bfloat16().requires_grad_(True)
    dout = torch.randn(B, S, Hq, D, device="cuda").bfloat16()
    torch.manual_seed(4)
    gen = torch.cuda.default_generators[torch.cuda.current_device()]
    seed, offset = gen.initial_seed(), gen.get_offset()
    o = prefix_lm_attention(q, k, v, P, dropout_p=p)
    o.backward(dout)
    assert gen.get_offset() == offset + ops.ATTN_DROPOUT_OFFSET_STEP
    keep = DR.attention_dropout_keep(seed, offset, B, Hq, S, p).cuda()
    t = lambda x: x.detach().transpose(1, 2)
    o_r, _, dq_r, dk_r, dv_r = DR.attention_ref_grouped_dropout(t(q), t(k), t(v), dout.transpose(1, 2), P, keep, p)
    assert rel_err(t(o), o_r) <= 1e-2
    assert rel_err(q.grad.transpose(1, 2), dq_r) <= 1e-2 and rel_err(k.grad.transpose(1, 2), dk_r) <= 1e-2
    assert rel_err(v.grad.transpose(1, 2), dv_r) <= 1e-2


def test_cuda_graph_capture_with_dropout_raises():
    B, S, H, D = 1, 128, 2, 128
    qkv = torch.randn(B * S, 3 * H * D, device="cuda").bfloat16()
    q, k, v = _split(qkv, H, H, D)
    ops.attn_fwd(q, k, v, B, S, H, H, D, 0)   # warm-up outside the capture
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with pytest.raises(NotImplementedError, match="CUDA-graph"):
            with torch.cuda.graph(g, stream=s):
                ops.attn_fwd(q, k, v, B, S, H, H, D, 0, dropout_p=0.1)
