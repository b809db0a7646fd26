"""Attention forward (and backward) throughput at the bench shapes, graph-replayed: TFLOP/s over unmasked pairs.
usage: [LLAMAX_B200_LIB=other.so] python tools/attn_fwd_perf.py [bwd] [sdpa] [dropout=P]
dropout=P: attention dropout at rate P (a fixed seed: the generator draw is not allowed in a graph capture); with sdpa,
SDPA runs at the same dropout_p."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from llamax_b200 import ops

import threading
import time

import pynvml

Hq, Hkv, D = 32, 8, 128
with_bwd = "bwd" in sys.argv[1:]
with_sdpa = "sdpa" in sys.argv[1:]   # also time cuDNN SDPA (causal configs) the same way
drop_p = float(next((a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("dropout=")), 0.0))
drop = dict(dropout_p=drop_p, rng=(1234, 0)) if drop_p > 0 else {}
pynvml.nvmlInit()
_h = pynvml.nvmlDeviceGetHandleByIndex(0)


class Clocks:
    """SM clock / power samples (NVML, every ~5 ms) while a timed loop runs."""

    def __enter__(self):
        self.s, self.p, self.on = [], [], True
        self.t = threading.Thread(target=self.run, daemon=True)
        self.t.start()
        return self

    def run(self):
        while self.on:
            self.s.append(pynvml.nvmlDeviceGetClockInfo(_h, pynvml.NVML_CLOCK_SM))
            self.p.append(pynvml.nvmlDeviceGetPowerUsage(_h) / 1e3)
            time.sleep(0.005)

    def __exit__(self, *a):
        self.on = False
        self.t.join()

    def summary(self):
        s = sorted(self.s)
        return f"SM {s[len(s) // 2]} MHz, {max(self.p):.0f} W" if s else "no samples"


def timeit(fn, n=5, reps=6):
    """(burst ms, sustained ms): best of n graph replays of `reps` calls, then the mean over a ~0.6 s back-to-back loop of
    the same graph at the power cap (the state the kernel runs in inside a training step), with NVML clocks / power."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / reps)
    global last_clocks
    k = max(3, int(600.0 / (min(ts) * reps)))
    for _ in range(k // 3):   # settle into the sustained state first
        g.replay()
    with Clocks() as c:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            g.replay()
        e1.record(); torch.cuda.synchronize()
    last_clocks = c.summary()
    return min(ts), e0.elapsed_time(e1) / (k * reps)


last_clocks = ""


for B, S, P in ((8, 2048, 0), (2, 8192, 0), (8, 1756, 1500), (4, 4096, 1024)):
    torch.manual_seed(0)
    ld = (Hq + 2 * Hkv) * D
    g = torch.randn(B * S, ld, device="cuda").bfloat16()
    q, k, v = g[:, : Hq * D], g[:, Hq * D : (Hq + Hkv) * D], g[:, (Hq + Hkv) * D :]
    pairs = S * P + (S - P) * (S - P + 1) / 2
    fl = 4.0 * B * Hq * D * pairs
    ms, sus = timeit(lambda: ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, P, **drop))
    line = f"B={B} S={S} P={P} dropout={drop_p}: fwd burst {fl / ms / 1e9:7.1f} sustained {fl / sus / 1e9:7.1f} TFLOP/s [{last_clocks}]"
    if with_bwd:
        o, lse = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, P, **drop)
        dout = torch.randn(B * S, Hq * D, device="cuda").bfloat16()
        dqkv = torch.empty_like(g)
        dq, dk, dv = dqkv[:, : Hq * D], dqkv[:, Hq * D : (Hq + Hkv) * D], dqkv[:, (Hq + Hkv) * D :]
        msb, susb = timeit(lambda: ops.attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, B, S, Hq, Hkv, D, P, **drop))
        line += f" | bwd burst {2.5 * fl / msb / 1e9:7.1f} sustained {2.5 * fl / susb / 1e9:7.1f} TFLOP/s [{last_clocks}]"
    print(line, flush=True)
    if with_sdpa and P == 0:
        import torch.nn.functional as F
        from torch.nn.attention import SDPBackend, sdpa_kernel

        q4 = q.view(B, S, Hq, D).transpose(1, 2).contiguous().requires_grad_(True)
        k4 = k.view(B, S, Hkv, D).transpose(1, 2).contiguous().requires_grad_(True)
        v4 = v.view(B, S, Hkv, D).transpose(1, 2).contiguous().requires_grad_(True)
        do4 = torch.randn(B, Hq, S, D, device="cuda").bfloat16()
        backends = [SDPBackend.CUDNN_ATTENTION] + ([SDPBackend.FLASH_ATTENTION, SDPBackend.EFFICIENT_ATTENTION]
                                                   if drop_p > 0 else [])
        with sdpa_kernel(backends):
            def f():
                return F.scaled_dot_product_attention(q4, k4, v4, is_causal=True, enable_gqa=True, dropout_p=drop_p)

            def fb():
                f().backward(do4)
                q4.grad = k4.grad = v4.grad = None

            try:
                ms, sus = timeit(f)
            except Exception as e:
                print(f"B={B} S={S} P={P} dropout={drop_p}: SDPA: {str(e)[:120]}", flush=True)
                continue
            line = f"B={B} S={S} P={P} dropout={drop_p}: SDPA fwd burst {fl / ms / 1e9:7.1f} sustained {fl / sus / 1e9:7.1f} TFLOP/s [{last_clocks}]"
            try:
                mfb, sfb = timeit(fb)
                line += f" | bwd (fwd+bwd - fwd) burst {2.5 * fl / (mfb - ms) / 1e9:7.1f} sustained {2.5 * fl / (sfb - sus) / 1e9:7.1f} TFLOP/s [{last_clocks}]"
            except Exception as e:   # autograd inside a graph capture may be refused
                line += f" | bwd: {str(e)[:80]}"
        print(line, flush=True)
