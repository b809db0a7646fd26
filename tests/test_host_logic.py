"""CPU: host-side logic of the drop-in seams (no kernels launched): subclass behaviour, module surgery, state-dict
compatibility with the reference, mask helpers, and loud failure off-GPU."""
import pytest
import torch
from torch import nn

from llamax_b200.modelling import (AudioConfig, Llama, LlamaAudio, LlamaConfig, LoRALinear, PrefixLM,
                                   apply_linear_adapter_)
from llamax_b200.modelling import llama as L
from llamax_b200.subclasses import Int8LinearWeight, int8_mm_dequant, quantize_int8_rowwise, quantize_linear_
from tests.helpers import load_golden


@pytest.fixture(scope="module")
def gold():
    return load_golden()


def test_from_float_matches_reference(gold):
    g = gold["int8_linear_dyn0"]
    W = Int8LinearWeight.from_float(g["w"], dynamic_int8_act=True)
    assert torch.equal(W.int_data, g["int_data"]) and torch.equal(W.scale, g["scale"])
    assert W.dtype is torch.bfloat16 and W.shape == g["w"].shape and W.dynamic_int8_act
    q, s = quantize_int8_rowwise(gold["quant"]["x"])
    assert torch.equal(q, gold["quant"]["q"]) and torch.equal(s, gold["quant"]["s"])


def test_subclass_dispatch_and_protocol(gold):
    g = gold["int8_linear_dyn0"]
    W = Int8LinearWeight(g["int_data"], g["scale"], True)
    d, c = W.detach(), W.clone()
    assert isinstance(d, Int8LinearWeight) and isinstance(c, Int8LinearWeight) and c.dynamic_int8_act
    assert c.int_data.data_ptr() != W.int_data.data_ptr()
    f = W.to(torch.float32)
    assert isinstance(f, Int8LinearWeight) and f.scale.dtype is torch.float32 and f.int_data.dtype is torch.int8
    names, attrs = W.__tensor_flatten__()
    W2 = Int8LinearWeight.__tensor_unflatten__({n: getattr(W, n) for n in names}, attrs)
    assert torch.equal(W2.int_data, W.int_data) and W2.dynamic_int8_act
    assert torch.equal(W.dequantize(), g["int_data"] * g["scale"].view(-1, 1))
    # copy_: subclass <- subclass, subclass <- float (re-quantise), float <- subclass
    dst = Int8LinearWeight(torch.zeros_like(g["int_data"]), torch.zeros_like(g["scale"]))
    dst.copy_(W)
    assert torch.equal(dst.int_data, W.int_data)
    dst2 = Int8LinearWeight(torch.zeros_like(g["int_data"]), torch.zeros_like(g["scale"]))
    dst2.copy_(g["w"])
    assert torch.equal(dst2.int_data, g["int_data"])
    flt = torch.zeros_like(g["w"])
    flt.copy_(W)
    assert torch.equal(flt, W.dequantize())
    with pytest.raises(NotImplementedError):
        W + 1  # anything outside detach / clone / to / copy_ is refused, like the reference


def test_linear_off_gpu_fails_loudly(gold):
    g = gold["int8_linear_dyn0"]
    W = Int8LinearWeight(g["int_data"], g["scale"], False)
    with pytest.raises(NotImplementedError, match="no CPU"):
        torch.nn.functional.linear(g["x"], W, None)
    with pytest.raises((NotImplementedError, RuntimeError)):
        int8_mm_dequant(torch.zeros(4, 16, dtype=torch.int8), torch.zeros(16, 8, dtype=torch.int8),
                        torch.ones(4, dtype=torch.bfloat16), torch.ones(8, dtype=torch.bfloat16))


def test_int8_mm_dequant_meta_and_asserts():
    A = torch.empty(32, 64, dtype=torch.int8, device="meta")
    B = torch.empty(48, 64, dtype=torch.int8, device="meta").T
    out = int8_mm_dequant(A, B, torch.empty(32, dtype=torch.bfloat16, device="meta"),
                          torch.empty(48, dtype=torch.bfloat16, device="meta"))
    assert out.shape == (32, 48) and out.dtype is torch.bfloat16
    with pytest.raises(AssertionError):
        int8_mm_dequant(A.to(torch.int16), B, torch.empty(32, device="meta"), torch.empty(48, device="meta"))


def _tiny():
    cfg = LlamaConfig(64, 2, 128, 2, 1, 128, max_seq_len=64, vocab_size=50, rope_base=500000, is_llama3_1=True)
    return LlamaAudio(cfg, AudioConfig(n_mels=80)).bfloat16()


def test_module_surgery_and_reference_state_dict(gold):
    model = _tiny()
    model.build_cache()
    quantize_linear_(model.layers, "int8", dynamic_int8_act=False)
    apply_linear_adapter_(model.layers, "lora", rank=8)
    wq = model.layers[0].attention.wq
    assert isinstance(wq, LoRALinear) and isinstance(wq.weight, Int8LinearWeight) and not wq.weight.requires_grad
    assert wq.lora_a.shape == (8, 64) and wq.lora_b.shape == (256, 8) and (wq.lora_b == 0).all() and wq.scale == 1.0
    assert isinstance(model.output.weight, nn.Parameter) and not isinstance(model.output.weight, Int8LinearWeight)
    ref_state = gold["audio_model"]["state"]
    assert set(model.state_dict().keys()) == set(ref_state.keys())  # same module / parameter names
    sd = {k: (Int8LinearWeight(v["int_data"], v["scale"]) if isinstance(v, dict) else v) for k, v in ref_state.items()}
    model.load_state_dict(sd)  # a reference checkpoint loads unchanged (copy_ dispatch on the subclass)
    k = "layers.1.feed_forward.w2.weight"
    assert torch.equal(model.state_dict()[k].int_data, ref_state[k]["int_data"])
    n_train = sum(p.numel() for p in model.layers.parameters() if p.requires_grad)
    assert n_train == sum(p.numel() for n, p in model.layers.named_parameters() if "lora" in n or "norm" in n)
    with pytest.raises(NotImplementedError):
        apply_linear_adapter_(_tiny(), "dora")


def test_rope_table_matches_reference(gold):
    cfg = LlamaConfig(128, 1, 64, 2, 1, 256, max_seq_len=48, rope_base=500000, is_llama3_1=False)
    assert torch.equal(L.build_rope(cfg), gold["rope_table_l31_0"]["table"])
    assert torch.equal(L.build_rope(cfg._replace(is_llama3_1=True)), gold["rope_table_l31_1"]["table"])
    assert torch.equal(L.build_rope(cfg._replace(is_llama3_1=True, head_dim=128, max_seq_len=16)),
                       gold["rope_table_hd128"]["table"])


def test_mask_plumbing():
    assert L._prefix_len_of(None, None, None) == 0
    assert L._prefix_len_of(None, PrefixLM(17), None) == 17
    assert L._prefix_len_of(torch.ones(4, 4, dtype=torch.bool), None, None) == 4    # fully bidirectional = prefix 4
    assert L._prefix_len_of(torch.ones(4, 4, dtype=torch.bool).tril(), None, None) == 0
    with pytest.raises(NotImplementedError):
        L._prefix_len_of(None, object(), None)
    with pytest.raises(NotImplementedError):
        L._prefix_len_of(None, None, torch.arange(4))
    model = _tiny()
    with pytest.raises(NotImplementedError):
        model.build_cache(inference=True)


def test_config_fields_match_reference():
    assert LlamaConfig._fields == ("embed_dim", "num_layers", "head_dim", "num_heads", "num_kv_heads",
                                   "intermediate_dim", "max_seq_len", "vocab_size", "attn_dropout", "rope_base",
                                   "is_llama3_1", "activation_checkpointing")
    assert AudioConfig()._asdict() == dict(sample_rate=16000, n_fft=512, win_length=400, hop_length=160, n_mels=128)


def test_gemm_tile_order_model_is_a_bijection():
    """tools/tile_order_model.py restates csrc/gemm.cu's tile_coords (both group orientations): every tile of a ragged
    grid is visited exactly once, and the orientation the launcher picks keeps no more panels live than the other."""
    import importlib.util
    import os

    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "tile_order_model.py")
    spec = importlib.util.spec_from_file_location("tile_order_model", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    for nm, nn in [(64, 16), (64, 56), (55, 16), (3, 5), (1, 1), (7, 501), (64, 4), (9, 9)]:
        for g in (8, -8, 3, -3):
            seen = {mod.coords(t, nm, nn, g) for t in range(nm * nn)}
            assert seen == {(a, b) for a in range(nm) for b in range(nn)}, (nm, nn, g)
    for nm, nn in [(64, 16), (55, 16), (32, 501), (64, 24)]:
        pick = -8 if nm >= nn else 8
        assert mod.live_panels(nm, nn, pick) <= mod.live_panels(nm, nn, -pick) + 1e-9


def test_dense_masks_and_block_masks_are_recognised():
    """Generic mask ingestion (SURVEY section 8(b)): dense boolean masks / FlexAttention mask_mods are compared with the
    prefix-LM and document-causal families rebuilt from the descriptor read off them; anything else raises."""
    import pytest

    from llamax_b200.modelling.llama import describe_dense_mask
    from oracle import ref_ops as R

    L = 96
    for P in (0, 1, 17, 96):
        d = describe_dense_mask(R.prefix_lm_mask(L, P))
        assert d.prefix_len == (0 if P <= 1 else P) and d.doc_start is None
    # one prefix length per sequence -> int32 [B]
    m = torch.stack([R.prefix_lm_mask(L, 5), R.prefix_lm_mask(L, 40)])[:, None]
    d = describe_dense_mask(m)
    assert d.prefix_len.tolist() == [5, 40]
    # packed documents
    doc_ids = torch.repeat_interleave(torch.arange(3), torch.tensor([30, 1, 65]))[None]
    d = describe_dense_mask(R.document_causal_mask(doc_ids))
    assert d.prefix_len == 0 and d.doc_start[0, 30].item() == 30 and d.doc_end[0, 29].item() == 29 and d.doc_start[0, 95].item() == 31
    # a sliding window is neither
    idx = torch.arange(L)
    with pytest.raises(NotImplementedError):
        describe_dense_mask((idx[:, None] >= idx[None, :]) & (idx[:, None] - idx[None, :] < 8))
    with pytest.raises(NotImplementedError):
        describe_dense_mask(torch.ones(L, L))          # not boolean


def test_bench_arms_share_one_config(monkeypatch):
    """bench.py: the GPU arm and `--impl reference` describe the same workload with the same `config` dict (one builder);
    the labelled-token count the reference arm states by formula equals the count of the synthetic batch."""
    import os
    import sys
    from types import SimpleNamespace

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)   # no CUDA driver in the CPU suite
    for batch, seq, gpus in ((8, 2048, 1), (8, 2048, 8), (2, 512, 2)):
        a = SimpleNamespace(layers=32, batch=batch, seq=seq, weight_only=False, rank=8, mixed_gemm=False,
                            int8_grad_input=False, gpus=gpus)
        host, positions, n_label = bench.make_batch(a, SimpleNamespace(vocab_size=128256), 0, "text")
        assert positions == batch * seq and n_label == bench.text_label_count(a)
        ours = bench.workload_config(a, gpus, "text", positions, n_label)
        ref = bench.workload_config(a, max(1, a.gpus), "text", a.batch * a.seq, bench.text_label_count(a))
        assert ours == ref and ours["parallelism"] == f"dp{gpus}" and ours["global_batch"] == batch * gpus
        assert "l2" in ours and ours["label_tokens_per_step"] == n_label * gpus


def test_bench_rejects_arguments_it_cannot_honour():
    """bench.py: fewer than one timed step, or an output dump from the CPU reference arm, is an argument error."""
    import os
    import subprocess
    import sys

    bench = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, bench, *extra], capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr)
