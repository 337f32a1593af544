"""Predictive uncertainty of WHVI classifiers on one GPU: what the entropy and log-predictive sums cost next to the predictive
sums they ride along with.

    python tools/bench_uncertainty.py [--reps 7] [--calls 50] [--warmup 3] [--out profiles/r08_uncertainty.json]

  * kernels: on the same (S, B, K) fp32 logits, ``whvi_categorical_uncertainty_f32`` (prob_sum, loglik_sum, logpred, ent_sum)
    against ``whvi_categorical_predictive_f32`` (prob_sum, loglik_sum), with labels, at (S, B, K) = (8, 512, 10), (8, 256, 1000),
    (64, 4096, 10), (16, 4096, 1000) and (4, 64, 65536): together they reach every work split of the kernel (TPR = 16 for
    K = 10, a warp per row for K = 1000, a CTA per row for K = 65536).  --reps blocks of --calls calls per arm, the arms
    alternating block by block, CUDA events around each block; the median block per call, in us, and the bytes/s achieved on
    the predictive's own algorithmic bytes (4 S B K of logits read once, the (B, K) sums written once, 8 B of labels and 4 B of
    loglik_sum per input) for both arms, so the two rates compare the same work.
  * networks: ``predictive_uncertainty`` against ``predict_proba`` on bench_classify's ``mnist`` and ``k1000`` models, 4096
    inputs x 64 samples in chunks of 16, fp32 and bf16 inputs, alternating, in inputs * samples per second.
Prints one JSON line and writes it to --out, with the card's name and power limit read (never set) in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from tools.bench_classify import EVAL_B, EVAL_CHUNK, EVAL_S, MODELS, _model, card  # noqa: E402

SHAPES = ((8, 512, 10), (8, 256, 1000), (64, 4096, 10), (16, 4096, 1000), (4, 64, 65536))


def _alternate(arms, calls, reps):
    """Median ms per call of each arm, the arms' blocks of ``calls`` calls interleaved rep by rep."""
    import torch
    blocks = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(calls):
                fn()
            b.record()
            b.synchronize()
            blocks[k].append(a.elapsed_time(b) / calls)
    return {k: (statistics.median(v), v) for k, v in blocks.items()}


def bench_kernels(args):
    import torch
    from whvi_b200 import functional as WF
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    rows = []
    for S, B, K in SHAPES:
        z = torch.randn((S, B, K), device=dev, generator=g) * 3
        y = torch.randint(0, K, (B,), device=dev, generator=g)
        prob, ent, ll, lp = (torch.empty(n, device=dev) for n in (B * K, B, B, B))
        arms = {"predictive": lambda: WF.categorical_predictive_(z, y, prob, ll),
                "uncertainty": lambda: WF.categorical_uncertainty_(z, y, prob, ent, ll, lp)}
        for fn in arms.values():
            for _ in range(args.warmup):
                fn()
        res = _alternate(arms, args.calls, args.reps)
        nbytes = 4 * S * B * K + 4 * B * K + 12 * B
        row = {"S": S, "B": B, "K": K, "predictive_bytes": nbytes}
        for k, (ms, blocks) in res.items():
            row[f"{k}_us"] = ms * 1e3
            row[f"{k}_GBps"] = nbytes / (ms * 1e-3) / 1e9
            row[f"{k}_blocks_ms"] = blocks
        row["overhead"] = row["uncertainty_us"] / row["predictive_us"] - 1.0
        rows.append(row)
    return rows


def bench_networks(args):
    import torch
    dev = torch.device("cuda:0")
    out = {}
    for name in args.models.split(","):
        dims, _ = MODELS[name]
        net = _model(dims)
        net.eval()
        g = torch.Generator(device=dev).manual_seed(1)
        x32 = torch.randn((EVAL_B, dims[0]), device=dev, generator=g)
        out[name] = {}
        for dt, x in (("fp32", x32), ("bf16", x32.to(torch.bfloat16))):
            arms = {"predict_proba": lambda: net.predict_proba(x, chunk_samples=EVAL_CHUNK),
                    "predictive_uncertainty": lambda: net.predictive_uncertainty(x, chunk_samples=EVAL_CHUNK)}
            for fn in arms.values():
                fn()
            res = _alternate(arms, 1, args.reps)
            row = {}
            for k, (ms, blocks) in res.items():
                row[f"{k}_ms"] = ms
                row[f"{k}_inputs_samples_per_s"] = EVAL_B * EVAL_S / (ms * 1e-3)
                row[f"{k}_blocks_ms"] = blocks
            row["overhead"] = row["predictive_uncertainty_ms"] / row["predict_proba_ms"] - 1.0
            out[name][dt] = row
        del net
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--models", default="mnist,k1000")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r08_uncertainty.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_uncertainty.py measures on a GPU; none is visible")
    out = {"card": card(), "reps": args.reps, "calls": args.calls,
           "eval": {"inputs": EVAL_B, "samples": EVAL_S, "chunk": EVAL_CHUNK},
           "kernels": bench_kernels(args), "networks": bench_networks(args)}
    print(json.dumps(out))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
