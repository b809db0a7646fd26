"""GPU: the deterministic training step (torch.use_deterministic_algorithms(True)).

With PyTorch's switch on, the attention backward takes dQ from attn_bwd_dq_kernel (fixed summation order in TMEM, no
fp32 atomics) and dK / dV from attn_bwd_kernel without its dQ^T product; lora_wgrad sums per-split partials in split
order; the LoRA backward takes the two-pass form (skinny dh GEMM + that lora_wgrad) instead of lora_bwd_pair; the
cross-entropy writes row losses that are summed in a fixed order. Checked here: parity against the fp64 oracle, dK / dV
bitwise equal to the default path, bitwise repeatability at sizes where many CTAs feed one output, which kernel classes
run with the switch on and off, and the tiny model under PyTorch's NaN fill of uninitialised memory.
"""
import pytest
import torch

from llamax_b200 import ops
from oracle import ref_ops as R
from tests.helpers import build_tiny_llama, oracle_layer_weights, rel_err
from tests.test_attention_gpu import CASES

pytestmark = pytest.mark.gpu


@pytest.fixture
def deterministic():
    """torch.use_deterministic_algorithms(True) with the NaN fill of torch.empty on; restored afterwards."""
    import torch.utils.deterministic as tud

    prev, prev_warn, prev_fill = (torch.are_deterministic_algorithms_enabled(),
                                  torch.is_deterministic_algorithms_warn_only_enabled(), tud.fill_uninitialized_memory)
    torch.use_deterministic_algorithms(True)
    tud.fill_uninitialized_memory = True
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
        tud.fill_uninitialized_memory = prev_fill


def _split(qkv, Hq, Hkv, Dh):
    return qkv[:, : Hq * Dh], qkv[:, Hq * Dh : (Hq + Hkv) * Dh], qkv[:, (Hq + Hkv) * Dh :]


def _bwd(qkv_dev, o, lse, dout_dev, B, S, Hq, Hkv, Dh, P, det, ds=None, de=None, rope=None):
    dqkv = torch.zeros_like(qkv_dev)
    dq, dk, dv = _split(dqkv, Hq, Hkv, Dh)
    ops.attn_bwd(*_split(qkv_dev, Hq, Hkv, Dh), o, lse, dout_dev, dq, dk, dv, B, S, Hq, Hkv, Dh, P, doc_start=ds,
                 doc_end=de, rope_inverse=rope, deterministic=det)
    return dq, dk, dv


# (B, S, Hq, Hkv, P, head_dim, document lengths): the fwd/bwd oracle cases, a per-sequence prefix vector, packed
# documents, head_dim 64
DQ_CASES = ([(B, S, Hq, Hkv, P, 128, None) for (B, S, Hq, Hkv, P) in CASES]
            + [(3, 300, 4, 2, [0, 77, 300], 128, None), (1, 640, 4, 1, 0, 128, [100, 28, 300, 212]),
               (1, 2048, 8, 2, 0, 128, [700, 1, 600, 747]), (2, 1024, 8, 2, 512, 64, None), (1, 300, 8, 2, 0, 64, None),
               (1, 129, 2, 1, 77, 64, None)])


@pytest.mark.parametrize("B,S,Hq,Hkv,P,Dh,lengths", DQ_CASES)
def test_deterministic_dq_vs_oracle_and_dkdv_bitwise(B, S, Hq, Hkv, P, Dh, lengths):
    torch.manual_seed(S + 11)
    qkv = torch.randn(B * S, (Hq + 2 * Hkv) * Dh).bfloat16()
    dout = torch.randn(B * S, Hq * Dh).bfloat16()
    q, k, v = _split(qkv, Hq, Hkv, Dh)
    to4 = lambda t, H, b: t.reshape(B, S, H, Dh)[b : b + 1].transpose(1, 2)
    doc_ids = ds = de = None
    if lengths is not None:
        doc_ids = torch.repeat_interleave(torch.arange(len(lengths)), torch.tensor(lengths))[None].expand(B, S).contiguous()
        ds, de = ops.doc_bounds(doc_ids.cuda())
    Pd = torch.tensor(P, device="cuda", dtype=torch.int32) if isinstance(P, list) else P
    g, gd = qkv.cuda(), dout.cuda()
    o, lse = ops.attn_fwd(*_split(g, Hq, Hkv, Dh), B, S, Hq, Hkv, Dh, Pd, doc_start=ds)
    dq0, dk0, dv0 = _bwd(g, o, lse, gd, B, S, Hq, Hkv, Dh, Pd, False, ds, de)
    dq1, dk1, dv1 = _bwd(g, o, lse, gd, B, S, Hq, Hkv, Dh, Pd, True, ds, de)
    assert torch.equal(dk1, dk0) and torch.equal(dv1, dv0)
    for b in range(B):
        Pb = P[b] if isinstance(P, list) else P
        _, dq_ref, _, _ = R.attention_ref_grads(to4(q, Hq, b), to4(k, Hkv, b), to4(v, Hkv, b), to4(dout, Hq, b), Pb,
                                                doc_ids=None if doc_ids is None else doc_ids[b : b + 1])
        assert rel_err(to4(dq1.cpu(), Hq, b), dq_ref) <= 1e-2


@pytest.mark.parametrize("Dh", [128, 64])
def test_deterministic_dq_rope_backward(Dh):
    """rope_inverse: the dQ kernel rotates its fp32 accumulator like attn_dq_convert_kernel does."""
    B, S, Hq, Hkv, P = 2, 384, 8, 2, 100
    torch.manual_seed(Dh)
    g = torch.randn(B * S, (Hq + 2 * Hkv) * Dh, device="cuda").bfloat16()
    gd = torch.randn(B * S, Hq * Dh, device="cuda").bfloat16()
    rope = R.build_rope(Dh, 512, 500000.0, True)[:S].contiguous().cuda()
    o, lse = ops.attn_fwd(*_split(g, Hq, Hkv, Dh), B, S, Hq, Hkv, Dh, P)
    dq0, dk0, dv0 = _bwd(g, o, lse, gd, B, S, Hq, Hkv, Dh, P, False, rope=rope)
    dq1, dk1, dv1 = _bwd(g, o, lse, gd, B, S, Hq, Hkv, Dh, P, True, rope=rope)
    assert torch.equal(dk1, dk0) and torch.equal(dv1, dv0)
    assert rel_err(dq1.float(), dq0.double()) <= 1e-2


def _wgrad_inputs():
    # P = 4096 -> 32 output tiles: the launcher splits the 16384 tokens over several CTAs per tile
    torch.manual_seed(4)
    X = torch.randn(16384, 4096, device="cuda").bfloat16()
    H = torch.randn(16384, 16, device="cuda").bfloat16()
    return X, H


def test_deterministic_lora_wgrad_vs_fp64():
    X, H = _wgrad_inputs()
    ref = 0.5 * (X.double().t() @ H.double())
    out = ops.lora_wgrad(X, H, 0.5, deterministic=True)
    assert out.dtype is torch.float32 and out.shape == (4096, 16)
    assert rel_err(out, ref) <= 1e-4


def _side_load(stop_after: int = 24):
    """Queue large GEMMs on a side stream: they compete for SMs with whatever runs next on the current stream."""
    s = torch.cuda.Stream()
    a = torch.randn(8192, 8192, device="cuda").bfloat16()
    with torch.cuda.stream(s):
        for _ in range(stop_after):
            ops.bf16_gemm(a, a)
    return s


@pytest.mark.parametrize("P", [0, 1024])
def test_attention_backward_repeatable(P):
    B, S, Hq, Hkv, Dh = 2, 4096, 32, 8, 128
    torch.manual_seed(P)
    g = torch.randn(B * S, (Hq + 2 * Hkv) * Dh, device="cuda").bfloat16()
    gd = torch.randn(B * S, Hq * Dh, device="cuda").bfloat16()
    o, lse = ops.attn_fwd(*_split(g, Hq, Hkv, Dh), B, S, Hq, Hkv, Dh, P)
    first = _bwd(g, o, lse, gd, B, S, Hq, Hkv, Dh, P, True)
    for run in range(3):
        side = _side_load() if run == 1 else None
        again = _bwd(g, o, lse, gd, B, S, Hq, Hkv, Dh, P, True)
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)
        for a, b in zip(first, again):
            assert torch.equal(a, b)


def test_lora_wgrad_repeatable():
    X, H = _wgrad_inputs()
    first = ops.lora_wgrad(X, H, 1.0, deterministic=True)
    for run in range(3):
        side = _side_load() if run == 1 else None
        assert torch.equal(ops.lora_wgrad(X, H, 1.0, deterministic=True), first)
        if side is not None:
            torch.cuda.current_stream().wait_stream(side)


def _tiny_step(model, tokens, labels, P):
    from llamax_b200.modelling import PrefixLM

    for p in model.parameters():
        p.grad = None
    loss = model(tokens, labels=labels, block_mask=PrefixLM(P))
    loss.backward()
    return loss.detach().clone(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}


def _tiny_model_case():
    dynamic, P, B, S = True, 64, 2, 192
    model = build_tiny_llama(dynamic, num_layers=4)
    cfg = model.config
    torch.manual_seed(5)
    tokens = torch.randint(0, cfg.vocab_size, (B, S))
    labels = torch.randint(0, cfg.vocab_size, (B, S))
    labels[:, :P] = -100
    return model, cfg, tokens, labels, P, dynamic


def test_tiny_model_step_repeatable(deterministic):
    model, cfg, tokens, labels, P, _ = _tiny_model_case()
    model = model.cuda()
    model.build_cache()
    model.tok_embeddings.requires_grad_(False)
    model.output.requires_grad_(False)
    tokens, labels = tokens.cuda(), labels.cuda()
    loss0, grads0 = _tiny_step(model, tokens, labels, P)
    assert len(grads0) > 0
    for _ in range(3):
        loss, grads = _tiny_step(model, tokens, labels, P)
        assert torch.equal(loss, loss0)
        assert grads.keys() == grads0.keys()
        for n in grads0:
            assert torch.equal(grads[n], grads0[n]), n


def test_tiny_model_loss_and_grads_deterministic(deterministic):
    """test_tiny_model_loss_and_grads with the switch on (and torch.empty filled with NaN): finite, same tolerances."""
    model, cfg, tokens, labels, P, dynamic = _tiny_model_case()
    S = tokens.shape[1]
    rope = R.build_rope(cfg.head_dim, cfg.max_seq_len, cfg.rope_base, cfg.is_llama3_1)[:S]
    lws = [oracle_layer_weights(l, torch.float32) for l in model.layers]
    x = model.tok_embeddings.weight.detach().float()[tokens]
    for lw in lws:
        x = R.transformer_layer_ref(x, rope, lw, cfg.num_heads, cfg.num_kv_heads, cfg.head_dim, P, dynamic)
    x = R.rmsnorm_ref(x, model.norm.weight.detach().float())
    logits = x @ model.output.weight.detach().float().T
    loss_ref = torch.nn.functional.cross_entropy(logits.view(-1, cfg.vocab_size), labels.view(-1))
    loss_ref.backward()

    model = model.cuda()
    model.build_cache()
    model.tok_embeddings.requires_grad_(False)
    model.output.requires_grad_(False)
    loss, grads = _tiny_step(model, tokens.cuda(), labels.cuda(), P)
    assert bool(torch.isfinite(loss)) and all(bool(torch.isfinite(g).all()) for g in grads.values())
    assert abs(loss.item() - loss_ref.item()) <= 2e-2 * abs(loss_ref.item()), (loss.item(), loss_ref.item())
    worst = 0.0
    for layer, lw in zip(model.layers, lws):
        att, ff = layer.attention, layer.feed_forward
        for name, mod in (("wq", att.wq), ("wo", att.wo), ("w1", ff.w1), ("w2", ff.w2)):
            worst = max(worst, rel_err(mod.lora_b.grad, lw.lora_b[name].grad))
    assert worst <= 5e-2


def _timed_classes(model, tokens, labels, P):
    ops.TIMING.enable()
    try:
        _tiny_step(model, tokens, labels, P)
        return set(ops.TIMING.summary())
    finally:
        ops.TIMING.disable()


def test_switch_selects_the_launches():
    model, cfg, tokens, labels, P, _ = _tiny_model_case()
    model = model.cuda()
    model.build_cache()
    model.tok_embeddings.requires_grad_(False)
    model.output.requires_grad_(False)
    tokens, labels = tokens.cuda(), labels.cuda()
    off = _timed_classes(model, tokens, labels, P)
    assert not any(c.endswith("_det") for c in off), off
    assert {"attn_bwd", "lora_wgrad", "cross_entropy"} <= off
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        on = _timed_classes(model, tokens, labels, P)
    finally:
        torch.use_deterministic_algorithms(prev)
    # lora_bwd_pair launches are timed as "lora_wgrad": neither it nor the atomic lora_wgrad may run
    assert "attn_bwd" not in on and "lora_wgrad" not in on and "cross_entropy" not in on, on
    assert {"attn_bwd_det", "lora_wgrad_det", "cross_entropy_det"} <= on


def test_8b_shape_block_repeatable(deterministic):
    """One decoder block at the Llama-3.1-8B shape (D 4096, F 14336, 32 / 8 heads, LoRA r = 8), 512 positions, prefix 300:
    output, input gradient and every parameter gradient identical over repeated runs."""
    from llamax_b200.modelling import LlamaConfig, PrefixLM

    cfg = LlamaConfig(4096, 1, 128, 32, 8, 14336, max_seq_len=512, vocab_size=1024, rope_base=500000, is_llama3_1=True)
    layer = build_tiny_llama(False, num_layers=1, config=cfg).layers[0].cuda()
    S = 512
    rope = R.build_rope(cfg.head_dim, cfg.max_seq_len, cfg.rope_base, cfg.is_llama3_1)[:S].cuda()
    torch.manual_seed(3)
    x = torch.randn(1, S, cfg.embed_dim, device="cuda").bfloat16()
    dout = torch.randn(1, S, cfg.embed_dim, device="cuda").bfloat16()

    def run():
        for p in layer.parameters():
            p.grad = None
        xc = x.clone().requires_grad_(True)
        out = layer(xc, rope, block_mask=PrefixLM(300))
        out.backward(dout)
        return [out.detach().clone(), xc.grad.clone()] + [p.grad.clone() for p in layer.parameters() if p.grad is not None]

    first = run()
    assert len(first) > 2
    for _ in range(2):
        again = run()
        assert len(again) == len(first)
        for a, b in zip(first, again):
            assert torch.equal(a, b)
