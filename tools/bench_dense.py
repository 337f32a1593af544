"""Diagonal against dense (full-covariance) posterior, in one process.

    python tools/bench_dense.py [--out FILE] [--c4-steps 3] [--c4-reps 3]

Workloads:
  * config 3 -- WHVIRegression [WHVILinear(13,128), ReLU, WHVILinear(128,128), ReLU, WHVILinear(128,1)], B = 4096, S = 64,
    loss + backward + Adam (torch.optim.Adam, capturable), eager and as one captured CUDA graph per step;
  * config 4 -- 3 x WHVILinear(4096,4096) with ReLUs, B = 8192, S = 128 in chunks of 32, loss + backward + FlatAdam
    (what bench.py times, diagonal arm);
  * device times of the dense C calls inside the config-3 dense step (Stacked D = 16, G = 8; square D = 128; Column
    D = 128; S = 64): the grouped reparameterisation forward and backward, the KL and the g-in / dg-out Stacked and Column calls.
Each pair of arms is warmed up, then timed in alternation (CUDA events around blocks of steps; the median block is
reported).  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import copy
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from tools.bench_bf16 import card  # noqa: E402


def _timed_blocks(fns, steps, reps):
    import torch
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                fn()
            b.record()
            torch.cuda.synchronize()
            times[k].append(a.elapsed_time(b) / steps)
    return {k: {"median": round(statistics.median(v), 4), "blocks": [round(t, 4) for t in v]} for k, v in times.items()}


def config3(dev):
    import torch
    import whvi_b200 as W
    from whvi_b200.graphs import GraphedTrainStep
    B, S = 4096, 64
    x, y = torch.randn(B, 13, device=dev), torch.randn(B, 1, device=dev)
    fns = {}
    for cov in ("diag", "dense"):
        torch.manual_seed(0)
        model = W.WHVIRegression([W.WHVILinear(13, 128, lambda_=3.0, covariance=cov), torch.nn.ReLU(),
                                  W.WHVILinear(128, 128, lambda_=3.0, covariance=cov), torch.nn.ReLU(),
                                  W.WHVILinear(128, 1, lambda_=3.0, covariance=cov)], train_samples=S).to(dev).train()
        graphed = copy.deepcopy(model)
        opt = torch.optim.Adam(model.parameters(), lr=torch.tensor(1e-3, device=dev), capturable=True)

        def step(model=model, opt=opt):
            model.loss(x, y, n=B).backward()
            opt.step()
            opt.zero_grad(set_to_none=True)

        opt_g = torch.optim.Adam(graphed.parameters(), lr=torch.tensor(1e-3, device=dev), capturable=True)
        gstep = GraphedTrainStep(graphed, opt_g, x, y, n=B)
        fns[f"{cov}:eager"] = step
        fns[f"{cov}:graph"] = lambda gstep=gstep: gstep(x, y)
    for fn in fns.values():
        for _ in range(5):
            fn()
    return {"workload": "config 3: 13-128-128-1, B=4096, S=64, loss + backward + Adam", "ms_per_step": _timed_blocks(fns, 20, 5)}


def config4(dev, steps, reps):
    import torch
    import whvi_b200 as W
    from whvi_b200.optim import FlatAdam, FlatParams
    D, B, S, chunk = 4096, 8192, 128, 32
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(B, D, generator=gen).to(dev)
    y = torch.randn(B, D, generator=gen).to(dev)
    fns, mem = {}, {}
    for cov in ("diag", "dense"):
        torch.manual_seed(0)
        model = W.WHVIRegression([W.WHVILinear(D, D, covariance=cov), torch.nn.ReLU(), W.WHVILinear(D, D, covariance=cov), torch.nn.ReLU(),
                                  W.WHVILinear(D, D, covariance=cov)], train_samples=chunk).to(dev).train()
        opt = FlatAdam(FlatParams(model.parameters()), lr=1e-3)

        def step(model=model, opt=opt):
            for _ in range(S // chunk):
                (model.loss(x, y, n=B) * (chunk / S)).backward()
            opt.step()
            opt.zero_grad()

        for _ in range(2):
            step()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        step()
        torch.cuda.synchronize()
        mem[cov] = round(torch.cuda.max_memory_allocated() / 2**30, 3)
        fns[cov] = step
    return {"workload": f"config 4: 3 x WHVILinear({D}) + ReLU, B={B}, S={S} in chunks of {chunk}, loss + backward + FlatAdam",
            "ms_per_step": _timed_blocks(fns, steps, reps), "peak_alloc_gib": mem}


NEW_CALLS = ("whvi_reparam_dense_grouped_f32", "whvi_reparam_dense_grouped_bwd_f32", "whvi_kl_dense_grouped_f32", "whvi_kl_dense_f32",
             "whvi_stacked_fwd_g_f32", "whvi_stacked_bwd_g_f32", "whvi_column_fwd_g_f32", "whvi_column_bwd_g_f32")


def kernels(dev, steps=20):
    """Device time of every dense C call inside the config-3 dense step (functional.EVENT_SINK: CUDA events on the launching
    stream around each call), median per call and shape."""
    import torch
    import whvi_b200 as W
    from whvi_b200 import functional as WF
    B, S = 4096, 64
    torch.manual_seed(0)
    model = W.WHVIRegression([W.WHVILinear(13, 128, lambda_=3.0, covariance="dense"), torch.nn.ReLU(),
                              W.WHVILinear(128, 128, lambda_=3.0, covariance="dense"), torch.nn.ReLU(),
                              W.WHVILinear(128, 1, lambda_=3.0, covariance="dense")], train_samples=S).to(dev).train()
    x, y = torch.randn(B, 13, device=dev), torch.randn(B, 1, device=dev)
    for _ in range(3):
        model.loss(x, y, n=B).backward()
    torch.cuda.synchronize()
    WF.EVENT_SINK = {c: [] for c in NEW_CALLS}
    for _ in range(steps):
        model.zero_grad(set_to_none=True)
        model.loss(x, y, n=B).backward()
    torch.cuda.synchronize()
    sink, WF.EVENT_SINK = WF.EVENT_SINK, None
    out = {}
    for call, recs in sink.items():
        by_tag = {}
        for a, b, tag in recs:
            by_tag.setdefault(tag, []).append(a.elapsed_time(b))
        for tag, ms in by_tag.items():
            out[f"{call} {tag}".strip()] = {"calls_per_step": len(ms) // steps, "us_median": round(1e3 * statistics.median(ms), 2)}
    return {"us_per_call": out, "timing": f"CUDA events around each call over {steps} eager config-3 dense steps (B={B}, S={S}): "
                                          "whvi_*_grouped at Stacked 13->128 (D=16, G=8) and at the square 128 and Column 128->1 "
                                          "layers (D=128, G=1)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c4-steps", type=int, default=3)
    ap.add_argument("--c4-reps", type=int, default=3)
    ap.add_argument("--out", type=Path, default=None, help="also write the JSON line here")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_dense.py needs a GPU"
    dev = torch.device("cuda", 0)
    res = {"card": card(), "config3": config3(dev), "kernels_config3_shapes": kernels(dev),
           "config4": config4(dev, args.c4_steps, args.c4_reps)}
    c3 = res["config3"]["ms_per_step"]
    c4 = res["config4"]["ms_per_step"]
    res["dense_over_diag"] = {"config3_eager": round(c3["dense:eager"]["median"] / c3["diag:eager"]["median"], 3),
                              "config3_graph": round(c3["dense:graph"]["median"] / c3["diag:graph"]["median"], 3),
                              "config4": round(c4["dense"]["median"] / c4["diag"]["median"], 3)}
    line = json.dumps(res)
    print(line)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
