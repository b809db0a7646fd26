"""Cost of the deterministic training step: bench.py's flagship text workload (Llama-3.1-8B, batch 8 x 2048, INT8 +
LoRA r = 8, one GPU) with torch.use_deterministic_algorithms off and on, alternated in one process on the same GPU.

    python tools/deterministic_ab.py [--steps 5] [--warmup 2] [--rounds 2]

Arms: "off"; "on" (PyTorch's default: torch.empty is also filled with NaN); "on_nofill"
(torch.utils.deterministic.fill_uninitialized_memory = False: the kernels' own cost). Per arm and round: resident-timed
ms/step and the per-step device time of the kernel classes that change (attention backward, LoRA weight gradients,
cross-entropy, bf16 GEMM, which also runs the two-pass LoRA dh), from bench.py's instrumented pass. Prints JSON lines;
the last one is the summary with the GPU name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CLASSES = ("attn_bwd", "attn_bwd_det", "lora_wgrad", "lora_wgrad_det", "cross_entropy", "cross_entropy_det", "bf16_gemm")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = (c.strip() for c in out.split(","))
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # the numbers are still device-timed; only the label is missing
        return {"gpu": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()

    import torch
    import torch.utils.deterministic as tud

    import bench

    sys.argv = ["bench.py", "--gpus", "1", "--steps", str(a.steps), "--warmup", str(a.warmup), "--workload", "text"]
    args = bench.parse()
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    arms = {"off": (False, True), "on": (True, True), "on_nofill": (True, False)}
    rows = []
    for rnd in range(a.rounds):
        for arm, (det, fill) in arms.items():
            torch.use_deterministic_algorithms(det)
            tud.fill_uninitialized_memory = fill
            try:
                res = bench.run_workload(args, "text", 0, 1, device, a.steps, a.warmup)
            finally:
                torch.use_deterministic_algorithms(False)
                tud.fill_uninitialized_memory = True
            kern = {k: round(v["ms"] / res["prof_steps"], 2) for k, v in res["kern"].items() if k in CLASSES}
            row = {"round": rnd, "arm": arm, "ms_per_step": round(res["ms"] / a.steps, 1),
                   "ms_per_step_e2e": round(res["ms_e2e"] / a.steps, 1), "loss": res["loss"], "kernel_ms_per_step": kern,
                   "sm_mhz": res["clocks"]["sm_mhz"] if res["clocks"] else None}
            rows.append(row)
            print(json.dumps(row), flush=True)
    summary = {"what": "deterministic mode A/B, Llama-3.1-8B text step, batch 8 x 2048, INT8 dynamic + LoRA r=8, 1 GPU",
               **gpu_info()}
    for arm in arms:
        ms = sorted(r["ms_per_step"] for r in rows if r["arm"] == arm)
        summary[f"{arm}_ms_per_step"] = ms
    summary["on_minus_off_ms_best"] = round(summary["on_ms_per_step"][0] - summary["off_ms_per_step"][0], 1)
    summary["on_nofill_minus_off_ms_best"] = round(summary["on_nofill_ms_per_step"][0] - summary["off_ms_per_step"][0], 1)
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
