"""Convolutional WHVI layers on one GPU: the patch kernels alone and a CNN classifier's training step.

    python tools/bench_conv.py [--steps 20] [--reps 5] [--warmup 3] [--out profiles/r07_conv.json]

  * patches: whvi_im2col_* and whvi_col2im_* on the two conv layers of the CNN below (S = 1: the shared first-layer input,
    and S = 8 for the second layer's per-sample input), fp32 and bf16, CUDA events over --steps * --reps calls (median
    block).  GB/s on the algorithmic bytes -- im2col: the patch matrix written plus the image read once; col2im: the n_in
    live columns of the patch gradient read plus dx written -- next to the copy rate measured in the same run (a 1 GiB
    device-to-device clone, read + write bytes).  The same tensors through torch: F.unfold + permute into the layer's column
    order (+ zero pad), and permute + F.fold.
  * step: synthetic 32 x 32 x 3 images, B = 128, S = 8 training samples, WHVIClassification
    [WHVIConv2d(3, 32, 3, padding=1), ReLU, MaxPool2d(2), WHVIConv2d(32, 64, 3, padding=1), ReLU, MaxPool2d(2), Flatten,
    WHVILinear(4096, 10)], FlatAdam; fp32 and bf16 images; eager and replayed as a captured CUDA graph (GraphedTrainStep).
    Step times from CUDA events (profiler off); kernel shares from a separate torch.profiler run of --steps steps (CUDA
    kernel time by kernel name, grouped), eager and graph.  For context only, the same architecture with deterministic
    nn.Conv2d / nn.Linear (cross-entropy, torch.optim.Adam), eager.
The second conv has n_in = 32 * 9 = 288 columns, padded to a D = 512 Stacked block and truncated to 64 outputs: each (sample,
pixel) row moves a D = 512 layer's bytes.  Prints one JSON line and writes it to --out, with the card's name and power limit
read in the same run.
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

B, S_TRAIN, N_DATA, K = 128, 8, 50000, 10


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
    return statistics.median(blocks)


def copy_rate(steps, reps):
    import torch
    src = torch.empty(1 << 28, dtype=torch.float32, device="cuda")   # 1 GiB: far beyond L2
    src.normal_()
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = _median_ms(lambda: dst.copy_(src), steps, reps)
    return 2 * src.numel() * 4 / ms / 1e6


def patch_arms(steps, reps, warmup):
    import torch
    import torch.nn.functional as F
    from whvi_b200 import functional as WF
    rows = []
    # (name, S, H, W, C, ld) with k = 3, padding 1: the CNN's two conv inputs
    for name, S, H, W, C, ld in (("conv1", 1, 32, 32, 3, 32), ("conv2", 1, 16, 16, 32, 512), ("conv2", S_TRAIN, 16, 16, 32, 512)):
        geom = (3, 3, 1, 1, 1, 1, 1, 1)
        n_in = C * 9
        for dtype in (torch.float32, torch.bfloat16):
            e = 2 if dtype == torch.bfloat16 else 4
            x = torch.randn((S, B, H, W, C), device="cuda").to(dtype)
            xi = x[0] if S == 1 else x
            N = B * H * W
            dp = torch.randn((S, N, ld), device="cuda").to(dtype)
            dpi = dp[0] if S == 1 else dp
            for _ in range(warmup):
                WF.im2col_(xi, geom, ld)
                WF.col2im_(dpi, geom, (B, H, W, C))
            im_ms = _median_ms(lambda: WF.im2col_(xi, geom, ld), steps, reps)
            c2_ms = _median_ms(lambda: WF.col2im_(dpi, geom, (B, H, W, C)), steps, reps)
            x_nchw = x.reshape(S * B, H, W, C).permute(0, 3, 1, 2).contiguous()

            def torch_unfold():
                u = F.unfold(x_nchw, 3, padding=1)                              # (S B, C 9, L): channel-major columns
                u = u.reshape(S * B, C, 9, H * W).permute(0, 3, 2, 1).reshape(S * B * H * W, n_in)
                return F.pad(u, (0, ld - n_in))

            dp_u = dp.reshape(S * B, H * W, ld)[..., :n_in]

            def torch_fold():
                u = dp_u.reshape(S * B, H * W, 9, C).permute(0, 3, 2, 1).reshape(S * B, n_in, H * W)
                return F.fold(u, (H, W), 3, padding=1).permute(0, 2, 3, 1).contiguous()

            for _ in range(warmup):
                torch_unfold()
                torch_fold()
            tu_ms = _median_ms(torch_unfold, steps, reps)
            tf_ms = _median_ms(torch_fold, steps, reps)
            im_bytes = S * N * ld * e + x.numel() * e
            c2_bytes = S * N * n_in * e + S * B * H * W * C * e
            rows.append({"layer": name, "S": S, "B": B, "H": H, "W": W, "C": C, "ld": ld, "dtype": str(dtype).split(".")[-1],
                         "im2col_ms": im_ms, "im2col_GBps": im_bytes / im_ms / 1e6, "torch_unfold_ms": tu_ms,
                         "col2im_ms": c2_ms, "col2im_GBps": c2_bytes / c2_ms / 1e6, "torch_fold_ms": tf_ms})
            del x, dp, x_nchw, dp_u
    return rows


def _data(dtype):
    import torch
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn((B, 3, 32, 32), device="cuda", generator=g).to(dtype)
    y = torch.randint(0, K, (B,), device="cuda", generator=g)
    return x, y


def whvi_net():
    import torch
    import torch.nn as nn
    import whvi_b200 as Wb
    torch.manual_seed(0)
    return Wb.WHVIClassification([Wb.WHVIConv2d(3, 32, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2), Wb.WHVIConv2d(32, 64, 3, padding=1),
                                  nn.ReLU(), nn.MaxPool2d(2), nn.Flatten(), Wb.WHVILinear(4096, K)], train_samples=S_TRAIN).cuda().train()


GROUPS = (("im2col", ("im2col_kernel",)), ("col2im", ("col2im_kernel",)),
          ("whvi_layer", ("layer_", "stack_", "column_", "reparam", "kl_", "bwd_reduce", "fwht")),
          ("categorical", ("categorical",)), ("adam", ("adam",)))


def kernel_shares(fn, steps):
    """CUDA kernel time per group of kernel names over ``steps`` calls of ``fn`` (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    per_name = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time > 0:
            per_name[ev.name] = per_name.get(ev.name, 0.0) + ev.device_time
    total = sum(per_name.values())
    groups = {g: 0.0 for g, _ in GROUPS}
    groups["other"] = 0.0
    for name, t in per_name.items():
        for g, keys in GROUPS:
            if any(k in name for k in keys):
                groups[g] += t
                break
        else:
            groups["other"] += t
    top = sorted(per_name.items(), key=lambda kv: -kv[1])[:12]
    return {"kernel_ms_per_step": total / steps / 1e3, "share": {g: t / total for g, t in groups.items()} if total else {},
            "top": [{"kernel": n[:120], "ms_per_step": t / steps / 1e3, "share": t / total} for n, t in top]}


def step_arms(steps, reps, warmup):
    import torch
    from whvi_b200 import FlatAdam, FlatParams
    from whvi_b200.graphs import GraphedTrainStep
    out = {}
    for dtype in (torch.float32, torch.bfloat16):
        x, y = _data(dtype)
        net = whvi_net()
        opt = FlatAdam(FlatParams(net.parameters()), lr=1e-3)

        def eager():
            loss = net.loss(x, y, n=N_DATA)
            loss.backward()
            opt.step()
            opt.zero_grad()

        for _ in range(warmup):
            eager()
        eager_ms = _median_ms(eager, steps, reps)
        eager_prof = kernel_shares(eager, steps)
        gnet = whvi_net()
        gopt = FlatAdam(FlatParams(gnet.parameters()), lr=1e-3)
        gstep = GraphedTrainStep(gnet, gopt, x, y, n=N_DATA)
        for _ in range(warmup):
            gstep(x, y)
        graph_ms = _median_ms(lambda: gstep(x, y), steps, reps)
        graph_prof = kernel_shares(lambda: gstep(x, y), steps)
        out[str(dtype).split(".")[-1]] = {"eager_ms": eager_ms, "graph_ms": graph_ms, "eager_kernels": eager_prof,
                                          "graph_kernels": graph_prof, "final_loss": float(net.loss(x, y, n=N_DATA))}
        del net, gnet, gstep, opt, gopt
    return out


def deterministic_arm(steps, reps, warmup):
    import torch
    import torch.nn as nn
    torch.manual_seed(0)
    net = nn.Sequential(nn.Conv2d(3, 32, 3, padding=1), nn.ReLU(), nn.MaxPool2d(2), nn.Conv2d(32, 64, 3, padding=1), nn.ReLU(),
                        nn.MaxPool2d(2), nn.Flatten(), nn.Linear(4096, K)).cuda()
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    x, y = _data(torch.float32)

    def eager():
        loss = nn.functional.cross_entropy(net(x), y)
        loss.backward()
        opt.step()
        opt.zero_grad()

    for _ in range(warmup):
        eager()
    return {"eager_ms": _median_ms(eager, steps, reps), "note": "torch nn.Conv2d / nn.Linear (cuDNN / cuBLAS), context only"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r07_conv.json"))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_conv needs a CUDA device")
    res = {"card": card(), "copy_GBps": copy_rate(a.steps, a.reps), "patches": patch_arms(a.steps, a.reps, a.warmup),
           "step": step_arms(a.steps, a.reps, a.warmup), "deterministic_cnn": deterministic_arm(a.steps, a.reps, a.warmup),
           "config": {"B": B, "S": S_TRAIN, "steps": a.steps, "reps": a.reps, "warmup": a.warmup}}
    line = json.dumps(res)
    print(line)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
