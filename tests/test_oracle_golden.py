"""CPU: the oracle restatement (oracle/ref_ops.py) against golden vectors produced by the reference code itself
(oracle/make_golden.py, run in the build container against /root/reference). Bit-exact wherever the oracle is the
same op sequence as the reference."""
import pytest
import torch

from oracle import ref_ops as R
from tests.helpers import load_golden


@pytest.fixture(scope="module")
def gold():
    return load_golden()


def test_quantize_rowwise_bit_exact(gold):
    g = gold["quant"]
    q, s = R.quantize_int8_rowwise(g["x"])
    assert torch.equal(q, g["q"]) and torch.equal(s, g["s"])
    assert (q[3] == 0).all() and s[3] == 0  # all-zero row: scale 0, codes 0 (clip 1e-12 path)


@pytest.mark.parametrize("dyn", [0, 1])
def test_int8_linear_fwd_bwd_bit_exact(gold, dyn):
    g = gold[f"int8_linear_dyn{dyn}"]
    q, s = R.quantize_int8_rowwise(g["w"])
    assert torch.equal(q, g["int_data"]) and torch.equal(s, g["scale"])
    y = R.int8_linear_fwd_ref(g["x"], g["int_data"], g["scale"], bool(dyn))
    assert torch.equal(y, g["y"])
    gx = R.int8_linear_bwd_ref(g["gout"], g["int_data"], g["scale"])
    assert torch.equal(gx, g["gx"])


def test_int8_mm_s32_is_exact():
    torch.manual_seed(0)
    A = torch.randint(-127, 128, (33, 64), dtype=torch.int8)
    B = torch.randint(-127, 128, (48, 64), dtype=torch.int8)
    assert torch.equal(R.int8_mm_s32(A, B.T), A.int() @ B.int().T)
    # adversarial range: K * 127^2 stays inside int32
    A = torch.full((17, 14336), 127, dtype=torch.int8)
    B = torch.full((8, 14336), -127, dtype=torch.int8)
    assert (R.int8_mm_s32(A, B.T) == -14336 * 127 * 127).all()


def test_lora_linear_matches_reference(gold):
    g = gold["lora_linear"]
    x = g["x"].clone().requires_grad_(True)
    a = g["lora_a"].clone().requires_grad_(True)
    b = g["lora_b"].clone().requires_grad_(True)
    y = R.Int8LinearRef.apply(x, g["int_data"], g["scale"], False) + R.lora_delta_ref(x, a, b, g["lora_scale"])
    assert torch.equal(y, g["y"])
    y.backward(g["gout"])
    assert torch.equal(x.grad, g["gx"]) and torch.equal(a.grad, g["ga"]) and torch.equal(b.grad, g["gb"])


def test_rope_tables_and_rotation(gold):
    assert torch.equal(R.build_rope(64, 48, 500000, False), gold["rope_table_l31_0"]["table"])
    assert torch.equal(R.build_rope(64, 48, 500000, True), gold["rope_table_l31_1"]["table"])
    assert torch.equal(R.build_rope(128, 16, 500000, True), gold["rope_table_hd128"]["table"])
    g = gold["apply_rope"]
    assert torch.equal(R.apply_rope(g["x"], g["table"]), g["y"])
    # inverse rotation undoes it up to bf16 rounding
    back = R.apply_rope_inverse(g["y"], g["table"])
    assert (back.float() - g["x"].float()).abs().max() < 0.05


def test_rmsnorm_and_swiglu_bit_exact(gold):
    g = gold["rmsnorm"]
    assert torch.equal(R.rmsnorm_ref(g["x"], g["w"]), g["y"])
    g = gold["swiglu"]
    assert torch.equal(R.swiglu_ref(g["a"], g["b"]), g["y"])


def _layer_weights(rec, dtype=torch.bfloat16):
    lw = R.LayerWeights()
    for n in R.LayerWeights.names:
        lw.w8[n], lw.ws[n] = rec[n]["int_data"], rec[n]["scale"].to(dtype)
        lw.lora_a[n] = rec[n]["lora_a"].to(dtype).clone().requires_grad_(True)
        lw.lora_b[n] = rec[n]["lora_b"].to(dtype).clone().requires_grad_(True)
    lw.lora_scale = rec["lora_scale"]
    lw.attention_norm = rec["an"].to(dtype).clone().requires_grad_(True)
    lw.ffn_norm = rec["fn"].to(dtype).clone().requires_grad_(True)
    return lw


@pytest.mark.parametrize("dyn", [0, 1])
def test_transformer_layer_matches_reference(gold, dyn):
    """Prefix-LM decoder block: forward bit-exact, gradients bit-exact (same op sequence, same autograd)."""
    rec = gold[f"layer_dyn{dyn}"]
    lw = _layer_weights(rec)
    x = rec["x"].clone().requires_grad_(True)
    c = rec["cfg"]
    out = R.transformer_layer_ref(x, rec["rope"], lw, c["Hq"], c["Hkv"], c["D"], rec["prefix_len"], bool(dyn))
    assert torch.equal(out, rec["out"])
    out.backward(rec["gout"])
    assert torch.equal(x.grad, rec["gx"])
    assert torch.equal(lw.attention_norm.grad, rec["g_an"]) and torch.equal(lw.ffn_norm.grad, rec["g_fn"])
    for n in R.LayerWeights.names:
        assert torch.equal(lw.lora_a[n].grad, rec[n]["ga"]), n
        assert torch.equal(lw.lora_b[n].grad, rec[n]["gb"]), n


def test_prefix_lm_mask_properties():
    m = R.prefix_lm_mask(10, 4)
    assert m[:, :4].all()                      # prefix visible to everyone
    assert torch.equal(m[4:, 4:], torch.tril(torch.ones(6, 6, dtype=torch.bool)))
    assert not m[0, 5]                         # prefix rows do not see the suffix
    assert torch.equal(R.prefix_lm_mask(7, 0), torch.tril(torch.ones(7, 7, dtype=torch.bool)))
    assert R.prefix_lm_mask(5, 9).all()        # P >= L: fully bidirectional


def test_attention_ref_matches_sdpa():
    torch.manual_seed(0)
    q, k, v = torch.randn(1, 4, 33, 16), torch.randn(1, 2, 33, 16), torch.randn(1, 2, 33, 16)
    ref = torch.nn.functional.scaled_dot_product_attention(q, k, v, R.prefix_lm_mask(33, 7), enable_gqa=True)
    assert torch.allclose(R.attention_ref(q, k, v, 7), ref, atol=1e-5)
