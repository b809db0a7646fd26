"""Pipeline-phase timeline of ONE attention-backward CTA (debug build with -DLX_ATTN_TRACE; SM-clock timestamps).

    python tools/attn_trace.py --build      # here (nvcc cross-compiles): csrc/libllamax_b200_trace.so
    python tools/attn_trace.py              # on the GPU box: prints per-step phase durations (cycles)
"""
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CSRC = os.path.join(ROOT, "llamax_b200", "csrc")
TRACE_LIB = os.path.join(CSRC, "libllamax_b200_trace.so")

if "--build" in sys.argv:
    from llamax_b200.build import FLAGS, NVCC, build
    build()
    obj = os.path.join(CSRC, "attention_trace.o")
    subprocess.check_call([NVCC, *FLAGS, "-DLX_ATTN_TRACE", "-c", os.path.join(CSRC, "attention.cu"), "-o", obj])
    others = [os.path.join(CSRC, f) for f in ("host_utils.o", "elementwise.o", "gemm.o")]
    subprocess.check_call([NVCC, "-shared", "-o", TRACE_LIB, obj, *others, "-gencode", "arch=compute_100a,code=sm_100a"])
    print("built", TRACE_LIB)
    sys.exit(0)

os.environ["LLAMAX_B200_LIB"] = TRACE_LIB
import torch  # noqa: E402

from llamax_b200 import _lib, ops  # noqa: E402

B, S, Hq, Hkv, D = 8, 2048, 32, 8, 128
P = int(os.environ.get("P", 0))
lib = _lib.load()
lib.llamax_debug_attn_trace.argtypes = [ctypes.c_void_p]
trace = torch.zeros(128 * 32, dtype=torch.int64, device="cuda")
assert lib.llamax_debug_attn_trace(trace.data_ptr()) == 0
ld = (Hq + 2 * Hkv) * D
g = torch.randn(B * S, ld, device="cuda").bfloat16()
q, k, v = g[:, : Hq * D], g[:, Hq * D : (Hq + Hkv) * D], g[:, (Hq + Hkv) * D :]
dout = torch.randn(B * S, Hq * D, device="cuda").bfloat16()
dqkv = torch.empty_like(g)
dq, dk, dv = dqkv[:, : Hq * D], dqkv[:, Hq * D : (Hq + Hkv) * D], dqkv[:, (Hq + Hkv) * D :]


def show(name, slots, first, last):
    t = trace.cpu().view(128, 32)
    t0 = int(t[first][slots[0][0]])
    print(f"== {name}: cycles since the first traced event; one row per step")
    print("step " + " ".join(f"{n:>9s}" for _, n in slots) + "   period")
    prev = None
    for s in range(first, last):
        row = [int(t[s][i]) - t0 if int(t[s][i]) else -1 for i, _ in slots]
        per = (row[0] - prev) if prev is not None else 0
        prev = row[0]
        print(f"{s:4d} " + " ".join(f"{x:9d}" for x in row) + f"   {per:6d}")


o, lse = ops.attn_fwd(q, k, v, B, S, Hq, Hkv, D, P)   # operands of the backward
for _ in range(2):
    ops.attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, B, S, Hq, Hkv, D, P)
torch.cuda.synchronize()
trace.zero_()
ops.attn_bwd(q, k, v, o, lse, dout, dq, dk, dv, B, S, Hq, Hkv, D, P)
torch.cuda.synchronize()
show("backward (CTA kv-tile 0, kv head 0): worker warp 4, drain warp 12, mma thread; step = 128 query rows",
     [(6, "w:top"), (7, "w:s_full"), (8, "w:S_regs"), (9, "w:p_arr"), (10, "w:dp_full"), (11, "w:ds_arr"),
      (12, "d:top"), (13, "d:dq_full"), (14, "d:in_reg"), (15, "d:end"),
      (0, "m:top"), (1, "m:p_full"), (2, "m:dV,S"), (3, "m:ds_full"), (4, "m:dQ,dK"), (5, "m:dP")],
     20, 44)
