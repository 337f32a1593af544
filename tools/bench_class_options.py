"""Class weights, label smoothing and ignore_index for WHVI classifiers on one GPU: what the options instances of the cross-entropy
kernels cost next to the plain ones.

    python tools/bench_class_options.py [--reps 7] [--calls 50] [--steps 20] [--warmup 3] [--out profiles/r09_class_options.json]

  * kernels: on the same (S, B, K) fp32 logits, at (S, B, K) = (8, 512, 10), (8, 256, 1000) and (4, 64, 65536) (TPR = 16, a
    warp per row, a CTA per row), the forward (``whvi_categorical_nll_f32``, two launches) and the backward
    (``whvi_categorical_nll_bwd_f32``) against ``whvi_categorical_nll_ex_f32`` / ``whvi_categorical_nll_bwd_ex_f32`` with
    weights, smoothing 0.1 and ignore_index -100 on every 8th row.  --reps blocks of --calls calls per arm, the arms alternating
    block by block, CUDA events around each block; the median block per call, in us.
  * steps: bench_conv's CNN classifier (two WHVIConv2d layers, a WHVILinear head, 128 CIFAR-sized images, 8 samples), one
    training step (loss, backward, FlatAdam) eager and replayed as a captured CUDA graph, with weights and smoothing 0.1 against
    the same step without them, the arms alternating; median ms per step.
Prints one JSON line and writes it to --out, with the card's name and power limit read (never set) in the same run.
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from tools.bench_classify import card  # noqa: E402
from tools.bench_conv import K as CNN_K, N_DATA, _data, whvi_net  # noqa: E402
from tools.bench_uncertainty import _alternate  # noqa: E402

SHAPES = ((8, 512, 10), (8, 256, 1000), (4, 64, 65536))


def bench_kernels(args):
    import torch
    from whvi_b200 import functional as WF
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    rows = []
    for S, B, K in SHAPES:
        z = (torch.randn((S, B, K), device=dev, generator=g) * 3).requires_grad_()
        y = torch.randint(0, K, (B,), device=dev, generator=g)
        y[::8] = -100
        yp = y.clamp(min=0)   # the plain call needs every label in range
        w = torch.rand(K, device=dev, generator=g) + 0.5
        opts = dict(weight=w, label_smoothing=0.1, ignore_index=-100)
        fwd = {"plain": lambda: WF.categorical_nll(z.detach(), yp), "options": lambda: WF.categorical_nll(z.detach(), y, **opts)}
        lp, lo = WF.categorical_nll(z, yp), WF.categorical_nll(z, y, **opts)
        one = torch.ones((), device=dev)
        bwd = {"plain": lambda: torch.autograd.grad(lp, z, one, retain_graph=True),
               "options": lambda: torch.autograd.grad(lo, z, one, retain_graph=True)}
        row = {"S": S, "B": B, "K": K}
        for what, arms in (("fwd", fwd), ("bwd", bwd)):
            for fn in arms.values():
                for _ in range(args.warmup):
                    fn()
            for k, (ms, blocks) in _alternate(arms, args.calls, args.reps).items():
                row[f"{what}_{k}_us"] = ms * 1e3
                row[f"{what}_{k}_blocks_ms"] = blocks
            row[f"{what}_overhead"] = row[f"{what}_options_us"] / row[f"{what}_plain_us"] - 1.0
        rows.append(row)
    return rows


def bench_steps(args):
    import torch
    import whvi_b200 as Wb
    from whvi_b200 import FlatAdam, FlatParams
    from whvi_b200.graphs import GraphedTrainStep
    x, y = _data(torch.float32)
    out = {}
    for mode in ("eager", "graph"):
        arms = {}
        for arm in ("plain", "options"):
            net = whvi_net()
            if arm == "options":
                net.likelihood = Wb.CategoricalLikelihood(weight=torch.linspace(0.5, 2.0, CNN_K), label_smoothing=0.1).cuda()
            opt = FlatAdam(FlatParams(net.parameters()), lr=1e-3)
            if mode == "graph":
                arms[arm] = (lambda s: lambda: s(x, y))(GraphedTrainStep(net, opt, x, y, n=N_DATA))
            else:
                def eager(net=net, opt=opt):
                    net.loss(x, y, n=N_DATA).backward()
                    opt.step()
                    opt.zero_grad()
                arms[arm] = eager
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        res = _alternate(arms, args.steps, args.reps)
        row = {f"{k}_ms": ms for k, (ms, _) in res.items()}
        row.update({f"{k}_blocks_ms": blocks for k, (_, blocks) in res.items()})
        row["overhead"] = row["options_ms"] / row["plain_ms"] - 1.0
        out[mode] = row
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r09_class_options.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_class_options.py measures on a GPU; none is visible")
    out = {"card": card(), "reps": args.reps, "calls": args.calls, "steps": args.steps,
           "kernels": bench_kernels(args), "cnn_step": bench_steps(args)}
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
