#!/usr/bin/env python
"""bench.py — train tokens/s of Llama-3.1-8B (frozen INT8 base + LoRA r=8) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload text|speech|both]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One JSON line on stdout (rank 0).  A "step" is one full optimizer step over one synthetic batch: forward, backward
through all 32 decoder blocks + LM head/cross-entropy, gradient all-reduce (N > 1), fused AdamW on the trainable
parameters.
  * headline (`value`, `e2e`, `roofline`, `kernels`): BASELINE.json `configs[1]` — MetaMathQA-shaped text SFT, causal
    (prefix length 0), batch 8 x 2048 per GPU.  `value` = whole-job positions/s with the batch resident in HBM; `e2e` =
    the same through the model's public forward with the batch in pinned host memory (H2D inside the timed region)
    and a D2H read of the loss every step.
  * `prefix_lm`: BASELINE.json `configs[2]` in the same line, same process, at every N — LibriSpeech-shaped 30 s audio ->
    1500-position bidirectional prefix + 256 text positions, prefix-LM mask, conv stem trainable (the DP payload grows
    from 42.5 to 145 MB).  Same two measurements + the attention kernels' rate on that mask.
  * `roofline` is the dominant kernel class (bf16 tcgen05 GEMM) on its heaviest shape; `roofline_int8` the INT8 GEMM on
    its heaviest shape against a cuBLASLt `torch._int_mm` 8192^3 peak measured in this process (outside every timed
    region), because MEASURED_PEAKS.json has no INT8 figure and the metric asks for "GEMM % INT8 peak".
`--impl reference` times the UNMODIFIED reference (baseline/_ref) on the host cores.
`--dump-outputs DIR` keeps the loss and gradients of the last timed step for comparing two builds output for output.
Batch and initial parameters are seeded and the optimizer runs at learning rate 0, so every step computes from the same
inputs. Float atomics (attention dQ, LoRA weight gradients, the loss sum) still make two runs agree to rounding, not bit
for bit: compare with a tolerance.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "train tokens/s, Llama-3.1-8B INT8+LoRA prefix-LM"
UNIT = "tokens/s"

LLAMA8B = dict(embed_dim=4096, num_layers=32, head_dim=128, num_heads=32, num_kv_heads=8, intermediate_dim=14336,
               vocab_size=128256, rope_base=500000, is_llama3_1=True)
# --dump-outputs: gradients kept per workload (float32, 16 MiB each; the speech step alone trains ~72 M parameters)
DUMP_GRADS = 1 << 22


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="both", choices=["text", "speech", "both"],
                    help="both: headline = text (configs[1]) + a `prefix_lm` record for speech (configs[2])")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--seq", type=int, default=2048)
    ap.add_argument("--layers", type=int, default=32)
    ap.add_argument("--weight-only", action="store_true", help="weight-only INT8 (bf16 GEMM) instead of dynamic")
    ap.add_argument("--rank", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-int8-peak", action="store_true")
    ap.add_argument("--cta-group", type=int, default=2)
    ap.add_argument("--ref-tokens", type=int, default=512, help="reference arm: positions of the bounded sample per step")
    ap.add_argument("--int8-grad-input", action="store_true",
                    help="OPT-IN, NON-PARITY: grad_input on the int8 tensor path (SURVEY 8 f4); never the headline")
    ap.add_argument("--mixed-gemm", action="store_true",
                    help="opt-in: mixed-input bf16 x int8 GEMMs (SURVEY K4/K5) for the weight-only forward and every "
                         "grad_input; identical results, no bf16 weight operands in HBM")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last resident-timed step of each workload computed as "
                         "DIR/<workload>_loss.npy (the loss) and DIR/<workload>_grads.npy (the trainable gradients after "
                         "the all-reduce, flattened in parameter order; a fixed seeded sample of %d of them where there "
                         "are more), float32" % DUMP_GRADS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        # median over the upper half of samples = under load (idle samples at the edges are dropped)
        busy = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ ours
def build_model(args, device, workload):
    import torch
    from llamax_b200.modelling import AudioConfig, Llama, LlamaAudio, LlamaConfig, apply_linear_adapter_
    from llamax_b200.subclasses import quantize_linear_

    cfgd = dict(LLAMA8B)
    cfgd["num_layers"] = args.layers
    cfgd["max_seq_len"] = 4096
    cfg = LlamaConfig(**cfgd)
    torch.manual_seed(1234)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device(device):
            model = LlamaAudio(cfg, AudioConfig(n_mels=80)) if workload == "speech" else Llama(cfg)
    finally:
        torch.set_default_dtype(prev)
    quantize_linear_(model.layers, "int8", dynamic_int8_act=not args.weight_only)
    apply_linear_adapter_(model.layers, "lora", rank=args.rank)
    g = torch.Generator(device=device).manual_seed(7)
    for m in model.modules():
        if hasattr(m, "lora_b"):  # non-zero B so that every backward GEMM does real work
            m.lora_b.data.normal_(0, 0.02, generator=g)
    model.tok_embeddings.requires_grad_(False)   # small-payload DP: only LoRA, norms (+ conv stem) train
    model.output.requires_grad_(False)
    model.build_cache()
    return model, cfg


def make_batch(args, cfg, rank, workload):
    """Synthetic MetaMathQA-shaped (text) or LibriSpeech-shaped (speech) batch in pinned host memory."""
    import torch

    g = torch.Generator().manual_seed(100 + rank)
    if workload == "text":
        tokens = torch.randint(0, cfg.vocab_size, (args.batch, args.seq), generator=g)
        labels = torch.roll(tokens, -1, 1)
        labels[:, : args.seq // 4] = -100   # prompt positions carry no loss
        labels[:, -1] = -100
        host = dict(tokens=tokens.pin_memory(), labels=labels.pin_memory())
        positions = args.batch * args.seq
    else:
        T = 256
        audio = torch.randn(args.batch, 480000, generator=g)  # 30 s @ 16 kHz -> 1500 prefix positions
        tokens = torch.randint(0, cfg.vocab_size, (args.batch, T), generator=g)
        labels = torch.roll(tokens, -1, 1)
        labels[:, -1] = -100
        host = dict(audio=audio.pin_memory(), tokens=tokens.pin_memory(), labels=labels.pin_memory())
        positions = args.batch * (1500 + T)
    n_label = int((host["labels"] != -100).sum())
    return host, positions, n_label


def load_ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed summary of an
    `ncu --set full` capture (profiles/ncu_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep); None if no
    capture of that kernel + shape has been committed."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        hit = table.get(kernel_key)
        return hit if hit is None else {"bytes": hit["bytes"], "source": hit.get("source"), "git": hit.get("git")}
    except Exception:
        return None


def measure_int8_peak(device):
    """cuBLASLt torch._int_mm 8192^3 (2*N^3 ops): best of 10 (burst) and back to back for ~3 s (sustained) — the same
    recipe MEASURED_PEAKS.json uses for bf16. A library call used only as the roofline DENOMINATOR, outside every timed
    region of the product path."""
    import torch

    n = 8192
    a = torch.randint(-127, 128, (n, n), device=device, dtype=torch.int8)
    b = torch.randint(-127, 128, (n, n), device=device, dtype=torch.int8).t()
    for _ in range(3):
        torch._int_mm(a, b)
    torch.cuda.synchronize()
    best = None
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
        t = e0.elapsed_time(e1)
        best = t if best is None or t < best else best
    reps = max(10, int(3000.0 / best))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch._int_mm(a, b)
    e1.record(); torch.cuda.synchronize()
    sus = e0.elapsed_time(e1) / reps
    ops_ = 2.0 * n ** 3
    return {"int8_tops": round(ops_ / best / 1e9, 1), "int8_tops_sustained": round(ops_ / sus / 1e9, 1),
            "how": "torch._int_mm (cuBLASLt) int8 8192^3, 2*N^3 ops: best of 10 (burst) and back to back for ~3 s (sustained)"}


def run_workload(args, workload, rank, world, device, steps, warmup):
    """Build the model of `workload`, run warm-up + resident-timed + e2e-timed + instrumented passes; returns a dict."""
    import torch
    import torch.distributed as dist

    from llamax_b200 import ops
    from llamax_b200.dp import GradBucket

    model, cfg = build_model(args, device, workload)
    params = [p for p in model.parameters() if p.requires_grad]
    # lr 0: the fused AdamW does the same work, but the parameters stay the seeded ones. With a real step size its
    # sign-like first updates turn the rounding noise of the float atomics into different parameters from run to run
    opt = torch.optim.AdamW(params, lr=0.0, weight_decay=0.0, fused=True)
    bucket = GradBucket(params)
    host, positions, n_label = make_batch(args, cfg, rank, workload)
    resident = {k: v.to(device) for k, v in host.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())
    dp_events, compute_events = [], []
    track = {"on": False}
    dump = None
    if args.dump_outputs:
        n_grad = sum(p.numel() for p in params)
        pick = None
        if n_grad > DUMP_GRADS:
            pick = torch.randperm(n_grad, generator=torch.Generator().manual_seed(0))[:DUMP_GRADS].sort().values
            pick = pick.to(device)
        dump = {"pick": pick}

    def step(batch, keep=None):
        if track["on"]:
            c0, c1, c2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            c0.record()
        if workload == "text":
            loss = model(batch["tokens"], labels=batch["labels"], block_mask=None)
        else:
            loss = model(batch["audio"], batch["tokens"], labels=batch["labels"], prefix_lm=True)
        loss.backward()
        if track["on"]:
            c1.record()
        bucket.allreduce_()
        if track["on"]:
            c2.record()
            compute_events.append((c0, c1))
            dp_events.append((c1, c2))
        if keep is not None:   # the gradients exist only until zero_grad below
            flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in params])
            keep["loss"] = loss.detach().clone()
            keep["grads"] = flat if keep["pick"] is None else flat[keep["pick"]]
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, e2e, keep=None):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for i in range(n):
            if e2e:
                batch = {k: v.to(device, non_blocking=True) for k, v in host.items()}
                last = step(batch).item()          # D2H read of the loss, every step
            else:
                last = step(resident, keep if i == n - 1 else None)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, (last if e2e else last.item())

    for _ in range(warmup):
        step(resident)
    barrier()

    sampler = ClockSampler(device.index)
    if rank == 0:
        sampler.start()
    # timed region: only the two GEMM classes (a few hundred launches) carry CUDA-event pairs, so the instrumentation
    # costs nothing measurable; the full per-kernel breakdown comes from a separate instrumented pass
    ops.TIMING.enable(only={"bf16_gemm", "int8_gemm"})
    track["on"] = world > 1
    ms, loss_val = timed(steps, e2e=False, keep=dump)
    kern_dom = ops.TIMING.summary()
    ops.TIMING.disable()
    track["on"] = False
    ms_e2e, _ = timed(steps, e2e=True)
    ops.TIMING.enable()
    prof_steps = min(steps, 5)
    ms_prof, _ = timed(prof_steps, e2e=False)
    kern = ops.TIMING.summary()            # every library launch, by kernel class (events around each: ~2 % overhead)
    ops.TIMING.disable()
    clocks = sampler.stop() if rank == 0 else None

    dp = None
    if world > 1:
        # where the DP time goes: (a) in-step all-reduce span (includes waiting for the slowest rank), (b) the collective
        # alone with the ranks aligned (pack + NCCL + unpack), (c) per-rank compute time per step (fwd + bwd, before the
        # all-reduce), gathered from every rank: the spread is the straggler effect
        in_step = sum(a.elapsed_time(b) for a, b in dp_events) / max(1, len(dp_events))
        comp = sum(a.elapsed_time(b) for a, b in compute_events) / max(1, len(compute_events))
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for p in params:
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        bucket.allreduce_()
        barrier()
        a0.record()
        for _ in range(10):
            bucket.allreduce_()
        a1.record()
        torch.cuda.synchronize()
        alone = a0.elapsed_time(a1) / 10
        t = torch.tensor([comp, in_step, alone], device=device)
        allr = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allr, t)
        comps = [float(x[0]) for x in allr]
        dp = {"dp_ms_per_step": round(max(float(x[1]) for x in allr), 3),
              "dp_ms_per_step_min_rank": round(min(float(x[1]) for x in allr), 3),
              "dp_collective_alone_ms": round(max(float(x[2]) for x in allr), 3),
              "compute_ms_per_rank": [round(c, 2) for c in comps],
              "compute_ms_spread": round(max(comps) - min(comps), 2),
              "note": "in-step all-reduce span = collective + waiting for the slowest rank's backward; "
                      "dp_collective_alone = pack + ncclAllReduce(AVG) + unpack with aligned ranks"}
        for p in params:
            p.grad = None

    res = dict(ms=ms, ms_e2e=ms_e2e, ms_prof=ms_prof, prof_steps=prof_steps, loss=loss_val, kern=kern,
               kern_dom=kern_dom, clocks=clocks, positions=positions, n_label=n_label, h2d_bytes=h2d_bytes,
               dp_payload=bucket.nbytes(), dp=dp, seq=(args.seq if workload == "text" else positions // args.batch))
    if dump is not None:
        res["dump"] = {k: dump[k].float().cpu().numpy() for k in ("loss", "grads")}
    del model, opt, bucket, params, resident, host
    gc.collect()
    torch.cuda.empty_cache()
    return res


def shape_table(kern, prefix, steps, peak):
    rows = []
    for k, v in kern.items():
        if k.startswith(prefix + "["):
            tf = v["flops"] / (v["ms"] / 1e3) / 1e12
            rows.append({"shape": k[len(prefix):], "launches_per_step": v["n"] // steps,
                         "ms_per_step": round(v["ms"] / steps, 2), "achieved": round(tf, 1),
                         "frac": round(tf / peak, 3) if peak else None})
    rows.sort(key=lambda r: -r["ms_per_step"])
    return rows


def run_ours(args):
    import torch
    import torch.distributed as dist

    from llamax_b200 import ops
    from llamax_b200.dp import init_distributed

    rank, world, local_rank = init_distributed()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    ops.set_gemm_cta_group(args.cta_group)
    if args.int8_grad_input:
        from llamax_b200.modelling import fused_block as _fb

        _fb.set_int8_grad_input(True)
    if args.mixed_gemm:
        from llamax_b200.modelling import fused_block as _fb

        _fb.set_mixed_gemm(True)
    warmup = max(args.warmup, 3)
    head_wl = "speech" if args.workload == "speech" else "text"
    main = run_workload(args, head_wl, rank, world, device, args.steps, warmup)
    pl = run_workload(args, "speech", rank, world, device, args.steps, warmup) if args.workload == "both" else None
    i8peak = None
    if rank == 0 and not args.no_int8_peak:
        i8peak = measure_int8_peak(device)

    if world > 1:
        dist.barrier()
        if rank != 0:
            dist.destroy_process_group()
    if rank != 0:
        return
    if args.dump_outputs:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for wl, r in ((head_wl, main), ("speech", pl)):
            for k, v in (r["dump"].items() if r is not None else ()):
                np.save(os.path.join(args.dump_outputs, f"{wl}_{k}.npy"), v)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    steps = args.steps
    positions, n_label = main["positions"], main["n_label"]
    assert head_wl != "text" or n_label == text_label_count(args)   # the reference arm states the same figure without a batch
    ms_step = main["ms"] / steps
    value = positions * world / (ms_step / 1e3)
    e2e_value = positions * world / (main["ms_e2e"] / steps / 1e3)
    kern_dom, kern_all = main["kern_dom"], main["kern"]
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1400"
    # dominant kernel = the bf16 tcgen05 GEMM; the roofline object is quoted on its heaviest shape (the w1|w3
    # grad_input GEMM, contraction over 2F + LoRA columns), timed live by CUDA events around each launch
    bf16_shapes = shape_table(kern_dom, "bf16_gemm", steps, peak_tf)
    i8_peak_sus = i8peak["int8_tops_sustained"] if i8peak else None
    int8_shapes = shape_table(kern_dom, "int8_gemm", steps, i8_peak_sus)
    roof = roof8 = None
    if bf16_shapes:
        dom = bf16_shapes[0]
        raw = kern_dom["bf16_gemm" + dom["shape"]]
        what = "grad_input of w1|w3" if "N=4096,K=28" in dom["shape"] else "largest bf16 GEMM of the step"
        kdim = int(dom["shape"].split("K=")[1].rstrip("]"))
        wide = kdim >= 8192 and args.cta_group == 2 and os.environ.get("LLAMAX_GEMM_WIDE", "1") != "0"
        key = ("gemm_wide_kernel<bf16,cta_group::2,512x256>%s" if wide else "gemm_kernel<bf16,cta_group::%d>%%s" % args.cta_group) % dom["shape"]
        tr = load_ncu_traffic(key)
        cls = kern_dom["bf16_gemm"]
        roof = {"kernel": "%s (%s)" % (key, what), "bound": "tensor", "achieved": dom["achieved"], "peak": peak_tf,
                "peak_source": peak_src, "unit": "TFLOP/s", "frac": round(dom["achieved"] / peak_tf, 4),
                "traffic": tr["bytes"] if tr else None, "traffic_source": (tr or {}).get("source"),
                "flops_per_launch": raw["flops"] / raw["n"], "us_per_launch": round(1e3 * raw["ms"] / raw["n"], 1),
                "launches_per_step": raw["n"] // steps, "ms_per_step": dom["ms_per_step"],
                "all_bf16_gemm_tflops": round(cls["flops"] / (cls["ms"] / 1e3) / 1e12, 1),
                "all_bf16_gemm_ms_per_step": round(cls["ms"] / steps, 2)}
    if int8_shapes:
        dom = int8_shapes[0]
        raw = kern_dom["int8_gemm" + dom["shape"]]
        cls = kern_dom["int8_gemm"]
        roof8 = {"kernel": "gemm_kernel<int8,cta_group::%d,lora8>%s (largest INT8 forward GEMM of the step)" % (args.cta_group, dom["shape"]),
                 "bound": "tensor", "achieved": dom["achieved"], "unit": "TOP/s",
                 "peak": i8_peak_sus, "frac": round(dom["achieved"] / i8_peak_sus, 4) if i8_peak_sus else None,
                 "peak_source": (i8peak["how"] + " — sustained figure, measured in this process after the timed regions; "
                                 "nominal dense INT8 4500") if i8peak else None,
                 "peak_burst": i8peak["int8_tops"] if i8peak else None,
                 "frac_of_nominal_4500": round(dom["achieved"] / 4500.0, 4),
                 "us_per_launch": round(1e3 * raw["ms"] / raw["n"], 1), "launches_per_step": raw["n"] // steps,
                 "ms_per_step": dom["ms_per_step"],
                 "all_int8_gemm_tops": round(cls["flops"] / (cls["ms"] / 1e3) / 1e12, 1),
                 "all_int8_gemm_ms_per_step": round(cls["ms"] / steps, 2)}

    def shares_of(kern, nsteps):
        flat = {k: v for k, v in kern.items() if "[" not in k}
        return {k: {"ms_per_step": round(v["ms"] / nsteps, 2), "launches_per_step": v["n"] // nsteps,
                    **({"achieved_tflops": round(v["flops"] / (v["ms"] / 1e3) / 1e12, 1)} if v.get("flops") else {}),
                    **({"achieved_gbs": round(v["bytes"] / (v["ms"] / 1e3) / 1e9, 1)} if v.get("bytes") else {})}
                for k, v in sorted(flat.items(), key=lambda kv: -kv[1]["ms"])}

    def launches_of(kern, nsteps):
        flat = {k: v for k, v in kern.items() if "[" not in k}
        return sum(v["n"] * (4 if k == "attn_bwd" else 2 if k == "lora_wgrad" else 1) for k, v in flat.items()) * steps // nsteps

    out = {
        "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(ms_step, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int8 fwd (int32 acc) / bf16 bwd" if not args.weight_only else "bf16 (int8 weights)",
        "data": "synthetic",
        "config": workload_config(args, world, head_wl, positions, n_label),
        "lm_head_rows": "final norm / LM head / cross-entropy run on the %d labelled rows per GPU and step only "
                        "(rows with label -100 contribute exact zeros to loss and gradients; identical results, "
                        "LLAMAX_LM_COMPACT=0 computes all %d rows)" % (n_label, positions),
        "label_tokens_per_s": round(n_label * world / (ms_step / 1e3), 1),
        "loss": round(float(main["loss"]), 4),
        "clocks": main["clocks"],
        "e2e": {"value": round(e2e_value, 1), "unit": UNIT, "h2d_bytes_per_step": main["h2d_bytes"], "d2h_bytes_per_step": 4,
                "ms_per_step": round(main["ms_e2e"] / steps, 2)},
        "gpu_launches": launches_of(kern_all, main["prof_steps"]),
        "roofline": roof,
        "roofline_int8": roof8,
        "kernels": shares_of(kern_all, main["prof_steps"]),
        "kernels_note": "per-class device time from a separate fully instrumented pass of the same steps (%.2f ms/step); "
                        "roofline, roofline_int8 and gemm_shapes are from the timed region itself" % (main["ms_prof"] / main["prof_steps"]),
        "gemm_shapes": {"bf16": bf16_shapes[:8], "int8": int8_shapes[:6]},
        "dp_payload_bytes": main["dp_payload"],
    }
    if main["dp"]:
        out["dp"] = main["dp"]
    if pl is not None:
        k = shares_of(pl["kern"], pl["prof_steps"])
        pls = pl["ms"] / steps
        out["prefix_lm"] = {
            "workload": workload_label(args, "speech", pl["positions"]),
            "value": round(pl["positions"] * world / (pls / 1e3), 1), "unit": "positions/s",
            "ms_per_step": round(pls, 2),
            "label_tokens_per_s": round(pl["n_label"] * world / (pls / 1e3), 1),
            "e2e": {"value": round(pl["positions"] * world / (pl["ms_e2e"] / steps / 1e3), 1), "unit": "positions/s",
                    "h2d_bytes_per_step": pl["h2d_bytes"], "d2h_bytes_per_step": 4,
                    "ms_per_step": round(pl["ms_e2e"] / steps, 2)},
            "seq_len": pl["seq"], "prefix_len": 1500, "positions_per_step": pl["positions"] * world,
            "attn_fwd_tflops": k.get("attn_fwd", {}).get("achieved_tflops"),
            "attn_bwd_tflops": k.get("attn_bwd", {}).get("achieved_tflops"),
            "attn_ms_per_step": round(k.get("attn_fwd", {}).get("ms_per_step", 0) + k.get("attn_bwd", {}).get("ms_per_step", 0), 2),
            "dp_payload_bytes": pl["dp_payload"], "loss": round(float(pl["loss"]), 4), "clocks": pl["clocks"],
            **({"dp": pl["dp"]} if pl["dp"] else {}),
        }
    if not args.no_cpu_baseline and world == 1:
        try:
            out["cpu_baseline"] = cpu_reference(args, steps=1, warmup=1)["baseline"]
        except Exception as e:  # the reference arm must never take the GPU line down with it
            out["cpu_baseline"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def workload_label(args, workload, positions=None):
    """`config.workload` of both arms (the reference arm times a bounded sample of the same workload)."""
    seq = args.seq if workload == "text" else (positions // args.batch if positions else 1500 + 256)
    return ("Llama-3.1-8B shape, frozen INT8 base + LoRA r=%d, %s, seq %d batch %d per GPU" %
            (args.rank, "MetaMathQA-shaped text SFT (causal)" if workload == "text"
             else "LibriSpeech-shaped 30 s audio prefix (1500) + 256 text, prefix-LM", seq, args.batch))


def text_label_count(args):
    """Labelled positions per GPU and step of the synthetic text batch (make_batch: the first quarter of every sequence
    is prompt, the last position has no successor)."""
    return args.batch * (args.seq - args.seq // 4 - 1)


def workload_config(args, world, workload, positions, n_label):
    """`config` of the JSON line: the workload only, identical for both arms (`--impl reference` times a bounded sample
    of exactly this workload on the host cores; what its sample is goes into its `cpu_baseline.sample`). Notes about
    how one arm computes the workload are top-level keys of that arm's line, not part of `config`."""
    cfg = {"workload": workload_label(args, workload, positions),
           "layers": args.layers, "global_batch": args.batch * world, "seq_len": positions // args.batch,
           "int8_mode": "weight-only" if args.weight_only else "dynamic_int8_act", "parallelism": f"dp{world}"}
    if args.mixed_gemm:
        cfg["mixed_gemm"] = "opt-in: bf16 x int8 mixed-input GEMMs (weights expanded inside the GEMM)"
    if args.int8_grad_input:
        cfg["NON_PARITY_OPT_IN"] = ("int8 grad_input (gradients quantised to 8 bit per row): not the reference's "
                                    "numerics, not a headline number")
    cfg["l2"] = "per-step working set (>10 GB activations + 7 GB weights) far exceeds the 126 MB L2; no flush needed"
    cfg["positions_per_step"] = positions * world
    cfg["label_tokens_per_step"] = n_label * world
    return cfg


# ------------------------------------------------------------------------------------------------ reference (CPU)
def cpu_reference(args, steps=1, warmup=1):
    """Time the UNMODIFIED reference (baseline/_ref: modelling.Llama, subclasses.quantize_linear_,
    modelling.apply_linear_adapter_) on the host cores, through its own public API `model(tokens, labels=labels)` +
    `loss.backward()`: Llama-3.1-8B shape, all 32 decoder blocks + final norm + LM head + cross-entropy, dynamic INT8 +
    LoRA r=8, causal (the text workload), on a BOUNDED sample of the batch: one sequence of `--ref-tokens` positions per
    step. The 32 entries of `model.layers` are ONE reference TransformerLayer (same module object 32 times): identical
    arithmetic per block, 0.2 GB instead of 7 GB of weights to initialise on the host. The only addition is the CPU
    registration of the reference's `torchao::int8_mm_dequant` op (baseline/ref_loader.py), which ships Meta + CUDA only.
    Falls back to the oracle port (kind "port") only if baseline/_ref is absent."""
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    S = int(args.ref_tokens)
    dynamic = not args.weight_only
    from baseline import ref_loader

    if ref_loader.available():
        modelling, subclasses = ref_loader.load(cpu_shim=True)
        cfgd = dict(LLAMA8B)
        cfgd["num_layers"] = 1
        cfgd["max_seq_len"] = max(S, 16)
        cfg = modelling.LlamaConfig(**cfgd)
        with torch.device("meta"):
            model = modelling.Llama(cfg)
        model = model.to_empty(device="cpu").bfloat16()
        with torch.no_grad():
            for p in model.parameters():
                if p.dim() > 1:
                    p.uniform_(-0.03, 0.03)
                else:
                    p.fill_(1.0)
        subclasses.quantize_linear_(model.layers, "int8", dynamic_int8_act=dynamic)
        modelling.apply_linear_adapter_(model.layers, "lora", rank=args.rank)
        with torch.no_grad():
            for m in model.modules():
                if hasattr(m, "lora_b"):
                    m.lora_b.normal_(0, 0.02)
        model.tok_embeddings.requires_grad_(False)
        model.output.requires_grad_(False)
        model.layers = torch.nn.ModuleList([model.layers[0]] * args.layers)   # one block's weights, applied 32 times
        model.build_cache()
        tokens = torch.randint(0, cfg.vocab_size, (1, S))
        labels = torch.roll(tokens, -1, 1)
        labels[:, : S // 4] = -100
        labels[:, -1] = -100
        kind = "reference"
        what = ("UNMODIFIED reference (baseline/_ref) on CPU, bf16, %s INT8 + LoRA r=%d: Llama-3.1-8B shape, %d blocks "
                "(one block's weights applied %d times) + norm + LM head + CE, fwd + bwd through model(tokens, labels=...), "
                "one sequence of %d positions per step (bounded sample of the 8 x 2048 batch; per-position CPU cost "
                "measured equal at 512 and 2048 positions: GEMM-bound)" %
                ("dynamic" if dynamic else "weight-only", args.rank, args.layers, args.layers, S))

        def one():
            t0 = time.perf_counter()
            loss = model(tokens, labels=labels)
            loss.backward()
            for p in model.parameters():
                p.grad = None
            return time.perf_counter() - t0
    else:
        from oracle import ref_ops as R

        D, Fd, Hq, Hkv, hd = 4096, 14336, 32, 8, 128
        lw = R.LayerWeights()
        shapes = dict(wq=(Hq * hd, D), wk=(Hkv * hd, D), wv=(Hkv * hd, D), wo=(D, Hq * hd), w1=(Fd, D), w3=(Fd, D), w2=(D, Fd))
        for n, (o, i) in shapes.items():
            lw.w8[n] = torch.randint(-127, 128, (o, i), dtype=torch.int8)
            lw.ws[n] = (torch.rand(o) * 1e-3).bfloat16()
            lw.lora_a[n] = (torch.randn(args.rank, i) * 0.02).bfloat16().requires_grad_(True)
            lw.lora_b[n] = (torch.randn(o, args.rank) * 0.02).bfloat16().requires_grad_(True)
        lw.attention_norm = torch.ones(D, dtype=torch.bfloat16, requires_grad=True)
        lw.ffn_norm = torch.ones(D, dtype=torch.bfloat16, requires_grad=True)
        rope = R.build_rope(hd, S, 500000, True)
        x0 = torch.randn(1, S, D).bfloat16().requires_grad_(True)
        w_out = (torch.randn(128256, D) * 0.02).bfloat16()
        labels = torch.randint(0, 128256, (S,))
        kind = "port"
        what = ("oracle port (baseline/_ref absent), PyTorch CPU bf16: 32 x one 8B-shape decoder block + LM head/CE on "
                "1 x %d positions per step" % S)

        def one():
            t0 = time.perf_counter()
            x = x0
            for _ in range(args.layers):
                x = R.transformer_layer_ref(x, rope, lw, Hq, Hkv, hd, 0, dynamic)
            loss = torch.nn.functional.cross_entropy((x.reshape(S, D) @ w_out.T).float(), labels)
            loss.backward()
            return time.perf_counter() - t0

    for _ in range(warmup):
        one()
    times = [one() for _ in range(max(steps, 1))]
    mean = sum(times) / len(times)
    base = {"value": round(S / mean, 2), "unit": UNIT, "cores": cores, "kind": kind, "sample": what,
            "seconds_per_step": round(mean, 3), "positions_per_step": S}
    return {"baseline": base, "times": times}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    r = cpu_reference(args, steps=args.steps, warmup=args.warmup)
    wall = time.perf_counter() - t0
    base = r["baseline"]
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * base["seconds_per_step"], 1),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16/int8 (CPU)",
           "data": "synthetic",
           "config": workload_config(args, max(1, args.gpus), "text", args.batch * args.seq, text_label_count(args)),
           "reference_sample": "bounded: one sequence of %d positions per step through all %d blocks + head (of the "
                               "%d x %d batch), host cores only" % (base["positions_per_step"], args.layers, args.batch,
                                                                    args.seq),
           "cpu_baseline": base,
           "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "wall_s": round(wall, 1)}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
