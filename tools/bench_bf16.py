"""Training steps with fp32 and with bf16 activations, in one process.

    python tools/bench_bf16.py [--model c4|c3|wide] [--steps 3] [--reps 3] [--warmup 2] [--chunk 32] [--out FILE]

--model c4 (default) is described below; the fp32 arm is what bench.py times.  The other two models are regression networks
that start with a Stacked layer and end with a transposed Column layer, and print their own JSON line (step time per arm, peak
allocation per arm, kernel launches per step, the card's name and power limit):
  * c3:   BASELINE config 3, [WHVILinear(13,128), ReLU, WHVILinear(128,128), ReLU, WHVILinear(128,1)], B = 4096, S = 64, full
          FlatAdam step, eager and captured as a CUDA graph (GraphedTrainStep).  Launch-bound: the step time says what bf16
          does to the launch count and host work, not to the bytes.
  * wide: [WHVILinear(13,4096), ReLU, WHVILinear(4096,4096), ReLU, WHVILinear(4096,1)], B = 8192, S = 128 in chunks of --chunk,
          eager, where the Stacked interleave and the Column kernels move enough bytes to be HBM-bound.  Also reports the
          per-call times of the Stacked and Column calls (functional.EVENT_SINK) with bytes/s on their algorithmic yardsticks:
          the activations each call must read and write once (Stacked forward: x + y; Stacked backward: x + dy, + dx when
          wanted; Column forward: x + y; Column backward: x + dy + dx), 2 bytes per bf16 and 4 per fp32 element, the
          transposed Column layer's y and dy always fp32.

Workload: BASELINE config 4 -- WHVIRegression of 3 x WHVILinear(4096, 4096) with ReLUs, B = 8192, S = 128 MC samples in
chunks of --chunk, forward + MNLL + KL + backward + FlatAdam -- once with an fp32 minibatch and once with the same
minibatch in bf16 (activations bf16 in HBM, parameters / gradients / arithmetic fp32).  Two copies of the model with
identical initial parameters, one per arm.  Both arms are warmed up, then timed in alternation (--reps blocks of --steps
steps each, CUDA events around each block; the median block is reported).

Prints one JSON line:
  * ms_per_step per arm (median and all blocks);
  * peak_alloc_gib per arm: torch.cuda.max_memory_allocated over one step, and the same minus what was allocated before it;
  * kernel times of the backward and loss-layer calls from functional.EVENT_SINK (one extra step per arm), per call
    position, with rates on their algorithmic yardsticks: backward (distinct x, with dx) x + dy + dx = 6 D bytes per row in
    bf16 (12 D in fp32), loss layer x + dx = 4 D bytes per row in bf16 (8 D in fp32; the target is shared by the samples);
  * the card's name and power limit, read in the same run.
"""
from __future__ import annotations

import argparse
import copy
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

D, B, S_TOTAL = 4096, 8192, 128
BWD_CALLS = ("whvi_layer_bwd_fused_f32", "whvi_layer_bwd_scaled_f32", "whvi_layer_bwd_bf16")
LOSS_CALLS = ("whvi_layer_loss_f32", "whvi_layer_loss_bf16")


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=10).stdout.strip()
        out["nvidia_smi"] = q
    except Exception as exc:   # reading the card's settings is informational
        out["nvidia_smi"] = f"unavailable: {exc}"
    return out


def _shapes_bench(args):
    """--model c3 / wide: fp32 and bf16 arms of a Stacked -> square -> Column regression network, timed in alternation."""
    import torch
    import whvi_b200 as W
    from whvi_b200 import functional as WF
    from whvi_b200.graphs import GraphedTrainStep
    from whvi_b200.optim import FlatAdam, FlatParams

    assert torch.cuda.is_available(), "bench_bf16.py needs a GPU"
    dev = torch.device("cuda", 0)
    c3 = args.model == "c3"
    n_in, width, batch, s_total = (13, 128, 4096, 64) if c3 else (13, 4096, 8192, 128)
    chunk = s_total if c3 else args.chunk
    n_chunks = s_total // chunk
    torch.manual_seed(0)
    base = W.WHVIRegression([W.WHVILinear(n_in, width), torch.nn.ReLU(), W.WHVILinear(width, width), torch.nn.ReLU(),
                             W.WHVILinear(width, 1)], train_samples=chunk).to(dev).train()
    gen = torch.Generator().manual_seed(1)
    x32 = torch.randn(batch, n_in, generator=gen).to(dev)
    y = torch.randn(batch, 1, generator=gen).to(dev)
    arms = {}
    for name, x in (("fp32", x32), ("bf16", x32.to(torch.bfloat16))):
        model = copy.deepcopy(base)
        flat = FlatParams(model.parameters())
        arms[name] = dict(model=model, opt=FlatAdam(flat, lr=torch.tensor(1e-3, device=dev)), x=x)
    del base

    def step(arm):
        m, opt = arm["model"], arm["opt"]
        for _ in range(n_chunks):
            loss = m.loss(arm["x"], y, n=batch)
            (loss * (1.0 / n_chunks) if n_chunks > 1 else loss).backward()
        opt.step()
        opt.zero_grad()

    modes = {"eager": step}
    if c3:
        for arm in arms.values():
            arm["graph"] = GraphedTrainStep(arm["model"], arm["opt"], arm["x"], y, n=batch)
        modes["graph"] = lambda arm: arm["graph"](arm["x"], y)

    def block(fn, arm, steps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn(arm)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    res_times = {}
    for mode, fn in modes.items():
        for arm in arms.values():
            for _ in range(args.warmup):
                fn(arm)
        times = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, arm in arms.items():
                times[k].append(block(fn, arm, args.steps))
        res_times[mode] = {k: {"median": round(statistics.median(v), 4), "blocks": [round(t, 4) for t in v]} for k, v in times.items()}
        res_times[mode]["bf16_over_fp32"] = round(statistics.median(times["bf16"]) / statistics.median(times["fp32"]), 4)

    memory, launches = {}, {}
    for k, arm in arms.items():
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        WF.LAUNCH_COUNTS.clear()
        step(arm)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        memory[k] = {"peak_alloc_gib": round(peak / 2**30, 3), "peak_minus_resident_gib": round((peak - before) / 2**30, 3)}
        launches[k] = {"library_launches_per_step": sum(WF.LAUNCH_COUNTS.values()), "by_call": dict(sorted(WF.LAUNCH_COUNTS.items()))}

    kernels = {}
    if not c3:
        calls = [f"whvi_{c}_{t}" for c in ("stacked_fwd", "stacked_bwd", "column_fwd", "column_bwd") for t in ("f32", "bf16")]
        for k, arm in arms.items():
            WF.EVENT_SINK = {c: [] for c in calls}
            step(arm)
            torch.cuda.synchronize()
            sink, WF.EVENT_SINK = WF.EVENT_SINK, None
            el = 2 if k == "bf16" else 4
            rows = chunk * batch
            for call, recs in sink.items():
                if not recs:
                    continue
                ms = [a.elapsed_time(b) for a, b, _ in recs]
                med = statistics.median(ms)
                if "stacked_fwd" in call:      # x (B, n_in) shared by the samples + y (S, B, width)
                    nbytes = el * (batch * n_in + rows * width)
                elif "stacked_bwd" in call:    # x + dy; the first layer's dx is not wanted
                    nbytes = el * (batch * n_in + rows * width)
                elif "column_fwd" in call:     # x (S, B, width) + y (S, B, 1) fp32
                    nbytes = el * rows * width + 4 * rows
                else:                          # x + dx + dy (S, B, 1) fp32
                    nbytes = 2 * el * rows * width + 4 * rows
                kernels[f"{k}:{call}"] = {"calls": len(ms), "ms_median": round(med, 4), "yardstick_bytes": nbytes,
                                          "TB_per_s_on_yardstick": round(nbytes / (med * 1e-3) / 1e12, 3)}

    res = {
        "workload": (f"{args.model} training step: WHVILinear({n_in},{width}) + ReLU + WHVILinear({width},{width}) + ReLU + "
                     f"WHVILinear({width},1), B={batch}, S={s_total}" + (f" in chunks of {chunk}" if n_chunks > 1 else "")
                     + ", fwd + MNLL + KL + bwd + FlatAdam"),
        "card": card(),
        "ms_per_step": res_times,
        "memory": memory,
        "launches": launches,
        "kernels": kernels,
        "timing": f"CUDA events around {args.reps} alternating blocks of {args.steps} steps per arm and mode after {args.warmup} "
                  "warm-up steps each; memory, launches and kernel times from further steps per arm",
    }
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", choices=("c4", "c3", "wide"), default="c4")
    ap.add_argument("--steps", type=int, default=3, help="steps per timed block")
    ap.add_argument("--reps", type=int, default=3, help="timed blocks per arm, alternating")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--chunk", type=int, default=32, help="MC samples per kernel launch")
    ap.add_argument("--out", type=Path, default=None, help="also write the JSON line here")
    args = ap.parse_args()
    if args.model != "c4":
        line = json.dumps(_shapes_bench(args))
        print(line)
        if args.out:
            args.out.parent.mkdir(parents=True, exist_ok=True)
            args.out.write_text(line + "\n")
        return

    import torch
    import whvi_b200 as W
    from whvi_b200 import functional as WF
    from whvi_b200.optim import FlatAdam, FlatParams

    assert torch.cuda.is_available(), "bench_bf16.py needs a GPU"
    dev = torch.device("cuda", 0)
    n_chunks = S_TOTAL // args.chunk
    torch.manual_seed(0)
    base = W.WHVIRegression([W.WHVILinear(D, D), torch.nn.ReLU(), W.WHVILinear(D, D), torch.nn.ReLU(), W.WHVILinear(D, D)],
                            train_samples=args.chunk).to(dev).train()
    gen = torch.Generator().manual_seed(1)
    x32 = torch.randn(B, D, generator=gen).to(dev)
    y = torch.randn(B, D, generator=gen).to(dev)
    arms = {}
    for name, x in (("fp32", x32), ("bf16", x32.to(torch.bfloat16))):
        model = copy.deepcopy(base)
        flat = FlatParams(model.parameters())
        arms[name] = dict(model=model, flat=flat, opt=FlatAdam(flat, lr=1e-3), x=x)
    del base

    def step(arm):
        m, opt = arm["model"], arm["opt"]
        for _ in range(n_chunks):
            (m.loss(arm["x"], y, n=B) * (1.0 / n_chunks)).backward()
        opt.step()
        opt.zero_grad()

    def block(arm, steps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            step(arm)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    for arm in arms.values():
        for _ in range(args.warmup):
            step(arm)
    times = {k: [] for k in arms}
    for _ in range(args.reps):
        for k, arm in arms.items():
            times[k].append(block(arm, args.steps))

    memory = {}
    for k, arm in arms.items():
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        step(arm)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated()
        memory[k] = {"peak_alloc_gib": round(peak / 2**30, 3), "peak_minus_resident_gib": round((peak - before) / 2**30, 3)}

    kernels = {}
    for k, arm in arms.items():
        WF.EVENT_SINK = {c: [] for c in BWD_CALLS + LOSS_CALLS}
        step(arm)
        torch.cuda.synchronize()
        sink, WF.EVENT_SINK = WF.EVENT_SINK, None
        el = 2 if k == "bf16" else 4
        rows = args.chunk * B
        for call, recs in sink.items():
            by_tag = {}
            for a, b, tag in recs:
                by_tag.setdefault(tag, []).append(a.elapsed_time(b))
            for tag, ms in by_tag.items():
                med = statistics.median(ms)
                e = {"calls": len(ms), "ms_median": round(med, 4)}
                if call in LOSS_CALLS and "nodx" not in tag:
                    e["yardstick_bytes_per_row"] = 2 * el * D
                elif call in BWD_CALLS and tag == "distinct_x":
                    e["yardstick_bytes_per_row"] = 3 * el * D
                if "yardstick_bytes_per_row" in e:
                    e["TB_per_s_on_yardstick"] = round(e["yardstick_bytes_per_row"] * rows / (med * 1e-3) / 1e12, 3)
                kernels[f"{k}:{call}:{tag}"] = e

    res = {
        "workload": f"config4 training step: 3x WHVILinear({D},{D})+ReLU, B={B}, S={S_TOTAL} in chunks of {args.chunk}, "
                    "fwd + MNLL + KL + bwd + FlatAdam",
        "card": card(),
        "ms_per_step": {k: {"median": round(statistics.median(v), 3), "blocks": [round(t, 3) for t in v]} for k, v in times.items()},
        "bf16_over_fp32_step_time": round(statistics.median(times["bf16"]) / statistics.median(times["fp32"]), 4),
        "memory": memory,
        "kernels": kernels,
        "timing": f"CUDA events around {args.reps} alternating blocks of {args.steps} steps per arm after {args.warmup} "
                  "warm-up steps each; kernel times from one further step per arm",
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
