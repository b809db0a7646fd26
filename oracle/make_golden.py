"""Generate the golden fixtures that pin the oracle (oracle/ref_ops.py) to the reference implementation.

Runs ONLY in the build container: imports the unmodified reference from /root/reference, executes its own code on
CPU with fixed seeds and stores small input/output vectors under tests/golden/.  The GPU box never sees
/root/reference; it only sees the committed fixtures.

    PYTHONPATH=/root/reference python oracle/make_golden.py

Reference entry points executed (file:line in the reference repo):
    subclasses/int8.py:10-16      quantize_int8_rowwise
    subclasses/int8.py:19-130     Int8LinearWeight.from_float, F.linear -> _Int8Linear fwd/bwd (weight-only; and
                                  dynamic through a 1-line CPU registration of torchao::int8_mm_dequant built on
                                  torch._int_mm — the reference ships only Meta/CUDA impls, int8_mm.py:135-149)
    modelling/lora.py:8-44        apply_linear_adapter_, LoRALinear.forward (+ autograd)
    modelling/llama.py:32-73      scale_llama3_1_rope, build_rope, apply_rope
    modelling/llama.py:143-174    FeedForward, TransformerLayer (SDPA branch with a dense prefix-LM mask)
    modelling/audio.py:38-77      LlamaAudio.forward (tiny config, prefix-LM via the causal_mask/input_pos hook)
"""
import io
import lzma
import os
import sys

import torch

REF = os.environ.get("LLAMAX_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")

import modelling  # noqa: E402  (reference)
import subclasses  # noqa: E402  (reference)
from modelling import llama as ref_llama  # noqa: E402
from subclasses import int8 as ref_int8  # noqa: E402
from subclasses import int8_mm as ref_int8_mm  # noqa: E402


@torch.library.impl(ref_int8_mm.lib, "int8_mm_dequant", "CPU")
def _cpu_int8_mm_dequant(A, B, a_scale, b_scale):
    # CPU stand-in for the Triton kernel: exact int32 accumulation, epilogue order of int8_mm.py:112-114
    return (torch._int_mm(A, B).float() * a_scale.float().view(-1, 1) * b_scale.float().view(1, -1)).to(a_scale.dtype)


def main():
    os.makedirs(OUT, exist_ok=True)
    g = {}
    torch.manual_seed(0)

    # ---- quantize_int8_rowwise
    x = (torch.randn(24, 256) * 3).bfloat16()
    x[3].zero_()
    q, s = ref_int8.quantize_int8_rowwise(x)
    g["quant"] = dict(x=x, q=q, s=s)

    # ---- Int8LinearWeight + _Int8Linear (both modes), forward and backward
    w = (torch.randn(96, 256) * 0.05).bfloat16()
    xin = torch.randn(2, 20, 256).bfloat16()
    gout = torch.randn(2, 20, 96).bfloat16()
    for dyn in (False, True):
        W = ref_int8.Int8LinearWeight.from_float(w, dynamic_int8_act=dyn)
        xi = xin.clone().requires_grad_(True)
        y = torch.nn.functional.linear(xi, W, None)
        y.backward(gout)
        g[f"int8_linear_dyn{int(dyn)}"] = dict(w=w, int_data=W.int_data, scale=W.scale, x=xin, y=y.detach(), gout=gout,
                                              gx=xi.grad)

    # ---- LoRALinear
    lin = torch.nn.Linear(256, 96, bias=False).bfloat16()
    lin.weight.data.copy_(w)
    subclasses.quantize_linear_(lin, "int8", dynamic_int8_act=False)
    modelling.apply_linear_adapter_(torch.nn.Sequential(lin), "lora", rank=8, alpha=16.0)
    lin.lora_b.data.copy_((torch.randn(96, 8) * 0.05).bfloat16())
    xi = xin.clone().requires_grad_(True)
    y = lin(xi)
    y.backward(gout)
    g["lora_linear"] = dict(int_data=lin.weight.int_data, scale=lin.weight.scale, lora_a=lin.lora_a.detach().clone(),
                            lora_b=lin.lora_b.detach().clone(), lora_scale=lin.scale, x=xin, y=y.detach(), gout=gout,
                            gx=xi.grad, ga=lin.lora_a.grad, gb=lin.lora_b.grad)

    # ---- RoPE
    for l31 in (False, True):
        cfg = ref_llama.LlamaConfig(128, 1, 64, 2, 1, 256, max_seq_len=48, rope_base=500000, is_llama3_1=l31)
        table = ref_llama.build_rope(cfg)
        g[f"rope_table_l31_{int(l31)}"] = dict(table=table)
    xr = torch.randn(2, 48, 3, 64).bfloat16()
    g["apply_rope"] = dict(x=xr, y=ref_llama.apply_rope(xr, table), table=table)
    cfg128 = ref_llama.LlamaConfig(128, 1, 128, 2, 1, 256, max_seq_len=16, rope_base=500000, is_llama3_1=True)
    g["rope_table_hd128"] = dict(table=ref_llama.build_rope(cfg128))

    # ---- RMSNorm / SwiGLU as the reference modules compute them
    norm = torch.nn.RMSNorm(256, eps=1e-5).bfloat16()
    norm.weight.data.copy_((1 + 0.1 * torch.randn(256)).bfloat16())
    xn = torch.randn(10, 256).bfloat16()
    g["rmsnorm"] = dict(x=xn, w=norm.weight.detach().clone(), y=norm(xn).detach())
    a, b = torch.randn(10, 64).bfloat16() * 2, torch.randn(10, 64).bfloat16()
    g["swiglu"] = dict(a=a, b=b, y=torch.nn.SiLU()(a) * b)

    # ---- one TransformerLayer, prefix-LM mask through the reference's SDPA branch, both INT8 modes
    cfg = ref_llama.LlamaConfig(128, 1, 128, 2, 1, 256, max_seq_len=160, vocab_size=64, rope_base=500000, is_llama3_1=True)
    L, P = 160, 50
    mask = (torch.arange(L)[None, :] < P) | (torch.arange(L)[:, None] >= torch.arange(L)[None, :])
    rope = ref_llama.build_rope(cfg)
    for dyn in (False, True):
        torch.manual_seed(1)
        layer = ref_llama.TransformerLayer(cfg).bfloat16()
        for n in (layer.attention_norm, layer.ffn_norm):
            n.weight.data.copy_((1 + 0.1 * torch.randn(128)).bfloat16())
        subclasses.quantize_linear_(layer, "int8", dynamic_int8_act=dyn)
        modelling.apply_linear_adapter_(layer, "lora", rank=8)
        for m in layer.modules():
            if hasattr(m, "lora_b"):
                m.lora_b.data.copy_((torch.randn(m.lora_b.shape) * 0.05).bfloat16())
        xl = torch.randn(1, L, 128).bfloat16().requires_grad_(True)
        gl = torch.randn(1, L, 128).bfloat16()
        out = layer(xl, rope[:L], mask=mask[None, None])
        out.backward(gl)
        rec = dict(x=xl.detach().clone(), gout=gl, out=out.detach(), gx=xl.grad, prefix_len=P,
                   cfg=dict(Hq=2, Hkv=1, D=128), an=layer.attention_norm.weight.detach().clone(),
                   fn=layer.ffn_norm.weight.detach().clone(), g_an=layer.attention_norm.weight.grad,
                   g_fn=layer.ffn_norm.weight.grad, rope=rope[:L].clone(), lora_scale=layer.attention.wq.scale)
        att, ff = layer.attention, layer.feed_forward
        for name, mod in (("wq", att.wq), ("wk", att.wk), ("wv", att.wv), ("wo", att.wo), ("w1", ff.w1), ("w3", ff.w3),
                          ("w2", ff.w2)):
            rec[name] = dict(int_data=mod.weight.int_data, scale=mod.weight.scale, lora_a=mod.lora_a.detach().clone(),
                             lora_b=mod.lora_b.detach().clone(), ga=mod.lora_a.grad, gb=mod.lora_b.grad)
        g[f"layer_dyn{int(dyn)}"] = rec

    # ---- tiny LlamaAudio end to end (config 1, downsized): loss with the prefix-LM mask hook
    from modelling import AudioConfig, LlamaAudio
    torch.manual_seed(2)
    cfg = ref_llama.LlamaConfig(64, 2, 128, 2, 1, 128, max_seq_len=64, vocab_size=50, rope_base=500000, is_llama3_1=True)
    model = LlamaAudio(cfg, AudioConfig(n_mels=80)).bfloat16()
    model.build_cache()
    subclasses.quantize_linear_(model.layers, "int8", dynamic_int8_act=False)
    modelling.apply_linear_adapter_(model.layers, "lora", rank=8)
    audio = torch.randn(1, 5120)                       # 0.32 s -> 33 frames -> 32 -> 16 prefix positions
    tokens = torch.randint(0, 50, (1, 24))
    labels = torch.randint(0, 50, (1, 24))
    Pn, Ltot = 16, 40
    model.register_buffer("causal_mask", (torch.arange(Ltot)[None, :] < Pn) | (torch.arange(Ltot)[:, None] >= torch.arange(Ltot)[None, :]), persistent=False)
    loss = model(audio, tokens, input_pos=torch.arange(Ltot), labels=labels)
    g["audio_model"] = dict(audio=audio, tokens=tokens, labels=labels, loss=loss.detach(), prefix_len=Pn,
                            state={k: (v if not isinstance(v, ref_int8.Int8LinearWeight) else dict(int_data=v.int_data, scale=v.scale))
                                   for k, v in model.state_dict().items()})

    path = os.path.join(OUT, "reference_vectors.pt.xz")
    buf = io.BytesIO()
    torch.save(g, buf)
    with open(path, "wb") as f:   # xz halves the 1.8 MB: many inputs repeat across records (tests/helpers.load_golden)
        f.write(lzma.compress(buf.getvalue(), preset=9 | lzma.PRESET_EXTREME))
    print("wrote", path, os.path.getsize(path) // 1024, "KiB;", "torch", torch.__version__)


if __name__ == "__main__":
    main()
