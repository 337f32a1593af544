"""Classification with WHVI networks on one GPU: training steps, the categorical likelihood's share of them, and predictive
evaluation.

    python tools/bench_classify.py [--steps 20] [--reps 5] [--warmup 3] [--out profiles/r06_classification.json]

Models (WHVIClassification, fp32 parameters, FlatAdam):
  * mnist:  [WHVILinear(784, 1024), ReLU, WHVILinear(1024, 1024), ReLU, WHVILinear(1024, 10)], B = 512, S = 8 training samples;
  * k1000:  [WHVILinear(784, 4096), ReLU, WHVILinear(4096, 4096), ReLU, WHVILinear(4096, 1000)], B = 256, S = 8.
Each model runs with an fp32 and with a bf16 minibatch (bf16 activations, so bf16 logits).  Per arm:
  * eager_ms / graph_ms: one training step (ELBO forward, backward, FlatAdam), eager and replayed as a captured CUDA graph
    (GraphedTrainStep); --reps blocks of --steps steps, CUDA events around each block, the median block per step;
  * likelihood_ms: CUDA-event time of the categorical forward and backward calls inside one eager step
    (functional.EVENT_SINK), and their share of eager_ms;
  * the same (S, B, K) logits through our kernels (CategoricalNLLFunction forward + backward) and through torch's
    log_softmax + gather + sum + autograd, each timed alone over --steps * --reps calls;
  * predictive: predict_proba over 4096 inputs x 64 samples in chunks of 16, in inputs * samples per second.
The logits are small next to the layers' activations (K = 10: 40 bytes per row), so these numbers say what the likelihood
costs a step, not what HBM can do.  Prints one JSON line and writes it to --out, with the card's name and power limit read in
the same run.
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

MODELS = {"mnist": ((784, 1024, 1024, 10), 512), "k1000": ((784, 4096, 4096, 1000), 256)}
S_TRAIN, N_DATA = 8, 60000
EVAL_B, EVAL_S, EVAL_CHUNK = 4096, 64, 16
LIK_CALLS = ("whvi_categorical_nll_f32", "whvi_categorical_nll_bf16", "whvi_categorical_nll_bwd_f32", "whvi_categorical_nll_bwd_bf16")


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        out["nvidia_smi"] = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                           capture_output=True, text=True, timeout=10).stdout.strip()
    except Exception as exc:   # reading the card's settings is informational
        out["nvidia_smi"] = f"unavailable: {exc}"
    return out


def _median_ms(fn, steps, reps):
    import torch
    blocks = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        b.synchronize()
        blocks.append(a.elapsed_time(b) / steps)
    return statistics.median(blocks), blocks


def _model(dims):
    import torch
    import torch.nn as nn
    import whvi_b200 as W
    torch.manual_seed(0)
    mods = []
    for i in range(len(dims) - 1):
        mods += [W.WHVILinear(dims[i], dims[i + 1], bias=True), nn.ReLU()]
    return W.WHVIClassification(mods[:-1], train_samples=S_TRAIN, eval_samples=EVAL_S).cuda()


def bench_arm(dims, B, bf16, args):
    import torch
    import whvi_b200 as W
    from whvi_b200 import functional as WF
    from whvi_b200.graphs import GraphedTrainStep
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn((B, dims[0]), device=dev, generator=g)
    x = x.to(torch.bfloat16) if bf16 else x
    y = torch.randint(0, dims[-1], (B,), device=dev, generator=g)
    res = {}

    eager = _model(dims)
    opt = W.FlatAdam(W.FlatParams(eager.parameters()), lr=1e-4)

    def eager_step():
        eager.loss(x, y, n=N_DATA).backward()
        opt.step()
        opt.zero_grad()

    for _ in range(args.warmup):
        eager_step()
    res["eager_ms"], res["eager_blocks"] = _median_ms(eager_step, args.steps, args.reps)

    WF.EVENT_SINK = {k: [] for k in LIK_CALLS}
    eager_step()
    torch.cuda.synchronize()
    lik = {k: sum(a.elapsed_time(b) for a, b, _ in v) for k, v in WF.EVENT_SINK.items() if v}
    WF.EVENT_SINK = None
    res["likelihood_ms"] = lik
    res["likelihood_share_of_eager_step"] = sum(lik.values()) / res["eager_ms"]

    graphed = _model(dims)
    opt_g = W.FlatAdam(W.FlatParams(graphed.parameters()), lr=1e-4)
    step = GraphedTrainStep(graphed, opt_g, x, y, n=N_DATA, warmup=args.warmup)
    res["graph_ms"], res["graph_blocks"] = _median_ms(lambda: step(x, y), args.steps, args.reps)
    del step, graphed, opt_g

    # the likelihood alone, ours against torch's, on the same logits
    with torch.no_grad():
        logits = eager._run(x, S_TRAIN).detach()
    S, Bq, K = logits.shape
    res["logits"] = {"shape": [S, Bq, K], "dtype": str(logits.dtype)}

    def ours():
        z = logits.requires_grad_()
        WF.categorical_nll(z, y).backward()
        z.grad = None

    def torch_ref():
        z = logits.requires_grad_()
        torch.log_softmax(z, -1).gather(-1, y.reshape(1, Bq, 1).expand(S, Bq, 1)).sum().neg().backward()
        z.grad = None

    for fn in (ours, torch_ref):
        for _ in range(args.warmup):
            fn()
    res["ours_fwd_bwd_ms"], _ = _median_ms(ours, args.steps * 5, args.reps)
    res["torch_fwd_bwd_ms"], _ = _median_ms(torch_ref, args.steps * 5, args.reps)

    # predictive evaluation: MC-mean probabilities, chunked
    eager.eval()
    xe = torch.randn((EVAL_B, dims[0]), device=dev, generator=g)
    xe = xe.to(torch.bfloat16) if bf16 else xe
    eager.predict_proba(xe, chunk_samples=EVAL_CHUNK)
    ms, _ = _median_ms(lambda: eager.predict_proba(xe, chunk_samples=EVAL_CHUNK), 1, args.reps)
    res["predictive_ms"] = ms
    res["predictive_inputs_samples_per_s"] = EVAL_B * EVAL_S / (ms * 1e-3)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--models", default="mnist,k1000")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_classification.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_classify.py measures on a GPU; none is visible")
    out = {"card": card(), "steps": args.steps, "reps": args.reps, "train_samples": S_TRAIN,
           "eval": {"inputs": EVAL_B, "samples": EVAL_S, "chunk": EVAL_CHUNK}, "models": {}}
    for name in args.models.split(","):
        dims, B = MODELS[name]
        out["models"][name] = {"dims": list(dims), "batch": B,
                               "fp32": bench_arm(dims, B, False, args), "bf16": bench_arm(dims, B, True, args)}
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
