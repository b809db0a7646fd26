"""Cost of attention dropout in the training step: bench.py's flagship text workload (Llama-3.1-8B, batch 8 x 2048,
INT8 + LoRA r = 8, one GPU) with LlamaConfig.attn_dropout 0 and 0.1, alternated in one process on the same GPU.

    python tools/attn_dropout_ab.py [--steps 5] [--warmup 2] [--rounds 2] [--p 0.1]

Per arm and round: resident-timed ms/step and the per-step device time of the attention kernel classes from bench.py's
instrumented pass (attn_fwd / attn_bwd without dropout, attn_fwd_drop / attn_bwd_drop with it). Prints JSON lines; the
last one is the summary with the GPU name and power limit.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.deterministic_ab import gpu_info  # noqa: E402

CLASSES = ("attn_fwd", "attn_bwd", "attn_fwd_drop", "attn_bwd_drop")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--p", type=float, default=0.1)
    a = ap.parse_args()

    import torch

    import bench

    sys.argv = ["bench.py", "--gpus", "1", "--steps", str(a.steps), "--warmup", str(a.warmup), "--workload", "text"]
    args = bench.parse()
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    build_model = bench.build_model
    arms = {"p0": 0.0, f"p{a.p:g}": a.p}
    rows = []
    for rnd in range(a.rounds):
        for arm, p in arms.items():
            def build(args_, device_, workload, p=p):
                model, cfg = build_model(args_, device_, workload)
                for layer in model.layers:
                    layer.attention.attn_dropout = p
                return model, cfg._replace(attn_dropout=p)

            bench.build_model = build
            try:
                res = bench.run_workload(args, "text", 0, 1, device, a.steps, a.warmup)
            finally:
                bench.build_model = build_model
            kern = {k: round(v["ms"] / res["prof_steps"], 2) for k, v in res["kern"].items() if k in CLASSES}
            row = {"round": rnd, "arm": arm, "ms_per_step": round(res["ms"] / a.steps, 1),
                   "ms_per_step_e2e": round(res["ms_e2e"] / a.steps, 1), "loss": res["loss"], "kernel_ms_per_step": kern,
                   "sm_mhz": res["clocks"]["sm_mhz"] if res["clocks"] else None}
            rows.append(row)
            print(json.dumps(row), flush=True)
    summary = {"what": f"attention dropout A/B (attn_dropout 0 vs {a.p:g}), Llama-3.1-8B text step, batch 8 x 2048, "
                       "INT8 dynamic + LoRA r=8, 1 GPU", **gpu_info()}
    for arm in arms:
        summary[f"{arm}_ms_per_step"] = sorted(r["ms_per_step"] for r in rows if r["arm"] == arm)
    keys = list(arms)
    summary["drop_minus_nodrop_ms_best"] = round(summary[f"{keys[1]}_ms_per_step"][0] - summary[f"{keys[0]}_ms_per_step"][0], 1)
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
