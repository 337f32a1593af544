#!/usr/bin/env python
"""bench.py -- the benchmark of the WHVI hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    (N > 1: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy (float32): `loss` (summed over
the ranks), `grad.<parameter>` (the all-reduced gradient the optimiser consumed) and `param.<parameter>` (the
parameters after its Adam update).  Inputs, parameters and noise are seeded, so two builds run with the same
arguments can be compared output for output.

Workload (BASELINE.json configs[3], the largest one that fits a single GPU): a wide WHVI
MLP of three WHVILinear(4096, 4096) layers with ReLU between them, minibatch B = 8192,
S = 128 MC samples => 2^20 (sample, row) pairs per layer per step.  One "step" = forward +
ELBO (Gaussian MNLL + KL) + backward of that model over the whole batch, plus the
parameter-gradient all-reduce (N > 1) and an Adam step.  MC samples are sharded across the
N GPUs (strong scaling: S stays 128) and processed in chunks of `--chunk` samples per
kernel launch so that activations stay at 4 GiB per tensor.

metric  = "WHVILinear fwd+bwd MC-sample rows/s": S*B*3 layer-rows / step time (a row = one
          (sample, minibatch-row) pair pushed through one WHVILinear forward AND backward).
value   = inputs resident in HBM;   e2e = same step, but x/y start in pinned host memory and
          the loss is read back to the host every step (through the public Python API).
Also in the line: `check` (loss and gradient checksum of ONE verification step on fixed noise -- identical
for every N up to summation order), the roofline of the dominant kernel (fused backward at a position
with per-sample inputs, 12*D algorithmic bytes per row) with every other kernel position beside it,
the batched-FWHT GB/s sweep over all ranks (`fwht`), the MC predictive-evaluation throughput of
BASELINE config 5 over all ranks (`eval`), and -- N = 1 only -- the CPU baseline.

`--impl reference`: the reference's OWN layer code (oracle/_ref/refpy, byte-compiled unmodified from
the reference sources by oracle/build.py) on the host cores: each step = one MC sample of one
WHVILinear(4096, 4096) over all 8192 rows, forward + backward.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

METRIC = "WHVILinear fwd+bwd MC-sample rows/s"
UNIT = "rows/s"
D_MODEL, B_BATCH, S_TOTAL, N_LAYERS = 4096, 8192, 128, 3
WORKLOAD = "config4-wide-mlp: 3x WHVILinear(4096,4096)+ReLU, B=8192, S=128 MC samples, fwd+bwd"
CONFIG = {"workload": WORKLOAD, "D": D_MODEL, "B": B_BATCH, "S": S_TOTAL, "layers": N_LAYERS}


def host_threads() -> int:
    return os.cpu_count() or 1


def use_all_host_threads() -> None:
    """torchrun exports OMP_NUM_THREADS=1 to every rank; a CPU leg that is supposed to use the host's cores
    must undo that BEFORE torch is imported (round 1 measured 80 instead of 350 rows/s with `cores: 32`)."""
    n = str(host_threads())
    os.environ["OMP_NUM_THREADS"] = n
    os.environ["MKL_NUM_THREADS"] = n


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# --------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.rows[0][1]),
                "reasons": reasons, "samples": len(self.rows)}


# --------------------------------------------------------------------------- CPU legs (the checker's code, never the product's)
def reference_layer_step_seconds():
    """One "reference step": ONE MC sample of ONE WHVILinear(4096, 4096) over ALL 8192 rows, forward + backward, on the
    host cores -- through the reference's own layer code when it travelled (kind "reference"), else through the
    torch-CPU restatement of it (kind "port").  Returns (seconds, kind)."""
    from oracle import ref_torch
    dt = ref_torch.reference_layer_fwd_bwd_seconds(D_MODEL, B_BATCH, 1)
    if dt is not None:
        return dt, "reference"
    return ref_torch.layer_fwd_bwd_seconds(D_MODEL, B_BATCH, 1), "port"


REF_SAMPLE = (f"each step = 1 of {S_TOTAL} MC samples x all {B_BATCH} rows x 1 of {N_LAYERS} layers, D={D_MODEL}, forward + backward, "
              f"on the host cores; rows/s = {B_BATCH} layer-rows / step time")


def cpu_layer_baseline(budget_s: float = 15.0):
    import torch
    torch.set_num_threads(host_threads())
    reference_layer_step_seconds()  # warm-up (allocator, H cache of the matmul path)
    t_used, done, kind = 0.0, 0, "port"
    while t_used < budget_s and done < 8:
        dt, kind = reference_layer_step_seconds()
        t_used += dt
        done += 1
    what = ("the reference's own WHVILinear (oracle/_ref/refpy: src/weights.py:66-93 byte-compiled unmodified)" if kind == "reference"
            else "torch CPU restatement of the reference layer as written (oracle/ref_torch.py)")
    return {"value": B_BATCH * done / t_used, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{done} step(s); {REF_SAMPLE}; {what}; {t_used:.1f} s of CPU work"}


def cpu_fwht_baseline():
    """The reference's own C++ CPU FWHT (oracle/_ref/fwht_cpp.so, compiled unmodified from
    src/fwht/cpp/fwht.cpp) if it travelled, else the C oracle port; D = 1024, 2^18 elements."""
    import torch
    from oracle import ref_torch
    torch.set_num_threads(host_threads())
    D, rows = 1024, 256
    mod = ref_torch.fwht_cpp_module()
    x = torch.randn(rows, D)
    if mod is not None:
        mod.forward(x[:8])
        t0 = time.perf_counter()
        mod.forward(x)
        dt = time.perf_counter() - t0
        kind = "reference"
    else:
        from oracle import oracle as O
        a = x.numpy()
        O.fwht(a[:8])
        t0 = time.perf_counter()
        O.fwht(a)
        dt = time.perf_counter() - t0
        kind = "port"
    return {"gbs": 8.0 * rows * D / dt / 1e9, "kind": kind, "D": D, "rows": rows, "cores": torch.get_num_threads(), "seconds": dt}


def gpu_fwht_reference_baseline(fwht_ours, dev, log2n: int = 28):
    """The reference's own CUDA FWHT (src/fwht/cuda, recompiled for sm_100a into oracle/_ref/fwht_cuda.so
    with the torch-API renames of SURVEY F3 only) timed on this GPU next to this repo's kernel, same
    inputs, through its public entry (which clones its input, fwht_cuda.cpp:11).  D <= 2^12 only: its
    launch shape is invalid beyond (SURVEY F2).  Baseline leg: one of the places bench.py may execute oracle/."""
    import torch
    from oracle import ref_torch
    mod = ref_torch.fwht_cuda_module()
    if mod is None:
        return None
    n = 1 << log2n
    x = torch.randn(n, device=dev)
    out = []
    for k in (6, 10, 12):
        Dk = 1 << k
        xv = x.view(n // Dk, Dk)
        try:
            got = mod.fwht(xv)
            ours = fwht_ours(xv)
            diff = float((got - ours).abs().max() / ours.abs().max())
            del got, ours
            for _ in range(2):
                mod.fwht(xv)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                mod.fwht(xv)
            b.record()
            b.synchronize()
            ms = a.elapsed_time(b) / 5
            out.append({"D": Dk, "ms": round(ms, 3), "gbs": round(8.0 * n / ms / 1e6, 1), "max_rel_diff_vs_ours": diff})
        except Exception as e:  # a baseline must never take the bench down
            out.append({"D": Dk, "error": str(e)[:120]})
    return {"kind": "reference CUDA kernel recompiled for sm_100a (oracle/_ref/fwht_cuda.so)", "elements": n, "sweep": out}


# --------------------------------------------------------------------------- reference arm
def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    use_all_host_threads()
    import torch
    torch.set_num_threads(host_threads())
    kind = "port"
    for _ in range(args.warmup):
        reference_layer_step_seconds()
    t = 0.0
    for _ in range(args.steps):
        dt, kind = reference_layer_step_seconds()
        t += dt
    value = B_BATCH * args.steps / t
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": dict(CONFIG),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": REF_SAMPLE},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def dump_outputs(out_dir, model, flat, loss, grad, world, rank):
    """--dump-outputs: the last timed step's loss, its all-reduced gradient and the parameters after its update, as
    float32 .npy files named after the parameters.  Every rank takes part in the loss all-reduce; rank 0 writes."""
    import numpy as np
    import torch.distributed as dist
    loss = loss.detach().clone()
    if world > 1:
        dist.all_reduce(loss)
    if rank != 0:
        return
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "loss.npy", loss.cpu().numpy())
    names = {id(p): name for name, p in model.named_parameters()}
    grad, param = grad.cpu().numpy(), flat.param.cpu().numpy()
    for p, off in zip(flat.params, flat.offsets):
        n = p.numel()
        np.save(out / f"grad.{names[id(p)]}.npy", grad[off:off + n].reshape(p.shape))
        np.save(out / f"param.{names[id(p)]}.npy", param[off:off + n].reshape(p.shape))


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    import whvi_b200 as W
    from whvi_b200 import functional as WF
    from whvi_b200 import fwht_
    from whvi_b200.distributed import shard_samples
    from whvi_b200.optim import FlatAdam, FlatParams

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # no NCCL_MAX_CTAS cap: the evaluation leg's pair exchange runs over peer memory without a collective kernel (its NCCL
        # fallback caps its own communicator), and the e2e leg's input all-gather wants its channels (0.7 -> 0.2 ms/step at N = 2)
        dist.init_process_group("nccl", device_id=dev)
    first_sample, S_local = shard_samples(S_TOTAL, rank, world)
    assert S_TOTAL % world == 0
    chunk = min(args.chunk, S_local)
    assert S_local % chunk == 0
    n_chunks = S_local // chunk
    D, B = D_MODEL, B_BATCH

    torch.manual_seed(0)  # parameters identical on every rank
    model = W.WHVIRegression([W.WHVILinear(D, D), torch.nn.ReLU(), W.WHVILinear(D, D), torch.nn.ReLU(),
                              W.WHVILinear(D, D)], train_samples=chunk).to(dev).train()
    # all parameters / gradients as views of two flat buffers: one memset, ONE all-reduce without pack/unpack
    # kernels, ONE fused Adam kernel per step (whvi_b200/optim.py)
    flat = FlatParams(model.parameters())
    opt = FlatAdam(flat, lr=1e-3)
    gen = torch.Generator().manual_seed(1)  # the same minibatch on every rank (MC-sample sharding)
    x_host = torch.randn(B, D, generator=gen).pin_memory()
    y_host = torch.randn(B, D, generator=gen).pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)
    scale = 1.0 / (n_chunks * world)
    blocks = [layer.square_blocks()[0] for layer in model._whvi_layers()]

    def fwd_bwd(x, y, eps=None):
        """Forward + ELBO + backward over this rank's sample shard in chunks; returns this rank's share of the loss.
        eps: per layer a (S_TOTAL, D) noise tensor to take this rank's rows from (verification), else fresh draws."""
        total = None
        for c in range(n_chunks):
            if eps is not None:
                lo = first_sample + c * chunk
                for blk, e in zip(blocks, eps):
                    blk.inject_eps(e[lo:lo + chunk])
            loss = model.loss(x, y, n=B) * scale
            loss.backward()
            total = loss.detach() if total is None else total + loss.detach()
        return total

    def step(x, y, grad_out=None):
        total = fwd_bwd(x, y)
        flat.all_reduce()  # one NCCL all-reduce on the flat gradient buffer (no-op at N = 1)
        if grad_out is not None:  # --dump-outputs: keep the gradient that zero_grad() is about to clear
            grad_out.copy_(flat.grad)
        opt.step()
        opt.zero_grad()
        return total

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        ms = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- verification step (before any training step: same parameters for every N): one GLOBAL noise tensor per
    # layer from a fixed seed, rank r takes sample rows [r S/N, (r+1) S/N); the summed loss and a checksum of the
    # all-reduced gradient must agree across N = 1, 2, 4, 8 up to fp32 summation order
    geps = torch.Generator().manual_seed(4242)
    eps_global = [torch.randn(S_TOTAL, D, generator=geps).to(dev) for _ in blocks]
    opt.zero_grad()
    check_loss = fwd_bwd(x_dev, y_dev, eps=eps_global).clone()
    flat.all_reduce()
    if world > 1:
        dist.all_reduce(check_loss)
    gcheck = flat.grad.double()
    wvec = torch.cos(torch.arange(gcheck.numel(), device=dev, dtype=torch.float64) * 0.37)
    check = {"loss": float(check_loss), "grad_l2": float(gcheck.norm()), "grad_dot_cos": float((gcheck * wvec).sum()),
             "note": "one step on fixed global eps (seed 4242), before training; must agree across n_gpus to ~1e-5 relative"}
    opt.zero_grad()
    del eps_global, gcheck, wvec

    # ---- warm-up, then the device-resident timed region -----------------------------------
    torch.manual_seed(100 + rank)  # timed steps: each rank draws its own eps shard
    import time
    for _ in range(max(args.warmup, 3)):
        step(x_dev, y_dev)
    # host time to ENQUEUE a step (empty launch queue at the start, no synchronisation inside: the GPU runs behind): the step
    # is GPU-bound while this stays below ms_per_step; at N = 8 the per-rank GPU work is 1/8, the host work per sample chunk is not
    torch.cuda.synchronize()
    t_host = time.perf_counter()
    step(x_dev, y_dev)
    step(x_dev, y_dev)
    host_enqueue_ms = (time.perf_counter() - t_host) * 1e3 / 2
    torch.cuda.synchronize()
    WF.LAUNCH_COUNTS.clear()
    timed_calls = ("whvi_layer_bwd_fused_f32", "whvi_layer_bwd_scaled_f32", "whvi_layer_fwd_fused_f32", "whvi_layer_loss_f32")
    WF.EVENT_SINK = {k: [] for k in timed_calls}
    last_grad = torch.empty_like(flat.grad) if args.dump_outputs else None
    losses = []

    def timed_step():
        final = len(losses) == args.steps - 1
        losses.append(step(x_dev, y_dev, last_grad if final else None))

    with ClockSampler(local_rank) as clk:
        ms_total = timed(timed_step, args.steps)
    sink, WF.EVENT_SINK = WF.EVENT_SINK, None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, model, flat, losses[-1], last_grad, world, rank)
    launches = sum(WF.LAUNCH_COUNTS.values())
    ms_step = ms_total / args.steps
    rows_per_step = S_TOTAL * B * N_LAYERS
    value = rows_per_step / (ms_step * 1e-3)

    # ---- end to end: pinned host inputs in, loss out, every step ---------------------------
    # Every step's x/y are copied from pinned host memory (a fresh H2D copy per step; N > 1: each rank copies 1/N of the
    # rows over its own PCIe link and the slices are all-gathered over NVLink) on a side stream while the previous step
    # computes (whvi_b200.utils.DevicePrefetcher), and every step's loss is copied to pinned host memory asynchronously:
    # the host reads loss i after it has launched step i+1, so the read-back never drains the GPU.
    from whvi_b200.utils import DevicePrefetcher
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    loss_ready = [torch.cuda.Event(), torch.cuda.Event()]

    def e2e_run(steps, verify=False):
        losses, pending = [], None
        for i, (x, y) in enumerate(DevicePrefetcher(((x_host, y_host) for _ in range(steps)), dev, shard_over_ranks=True)):
            if verify:   # warm-up only: what the ranks handed each other over NVLink is the minibatch, bit for bit
                assert torch.equal(x, x_dev) and torch.equal(y, y_dev), "DevicePrefetcher delivered a different minibatch"
            total = step(x, y)
            loss_host[i % 2].copy_(total, non_blocking=True)
            loss_ready[i % 2].record()
            if pending is not None:
                loss_ready[pending].synchronize()
                losses.append(float(loss_host[pending]))
            pending = i % 2
        if pending is not None:
            loss_ready[pending].synchronize()
            losses.append(float(loss_host[pending]))
        return losses

    e2e_run(3, verify=True)
    e2e_losses = []
    ms_e2e = timed(lambda: e2e_losses.extend(e2e_run(args.steps)), 1) / args.steps
    e2e_value = rows_per_step / (ms_e2e * 1e-3)
    assert len(e2e_losses) == args.steps and all(l == l for l in e2e_losses)

    # ---- roofline per kernel position, from CUDA events recorded around the calls inside the timed region -------------
    peak, peak_src = measured_peaks()
    rows_per_launch = chunk * B

    def position(calls, tag, alg_bytes_per_row, dram_note):
        tags = tag if isinstance(tag, tuple) else (tag,)
        ms = [a.elapsed_time(b) for name in calls for a, b, t in sink[name] if t in tags]
        if not ms:
            return None
        avg = sum(ms) / len(ms)
        gbs = alg_bytes_per_row * rows_per_launch / (avg * 1e-3) / 1e9
        return {"achieved": gbs, "frac": gbs / peak, "frac_of_8TBs_nominal": gbs / 8000.0, "avg_launch_ms": avg, "launches_timed": len(ms),
                "algorithmic_bytes_per_row": alg_bytes_per_row, "share_of_step": sum(ms) / ms_total, "expected_dram_bytes_per_row": dram_note}

    bwd_calls = ("whvi_layer_bwd_fused_f32", "whvi_layer_bwd_scaled_f32")
    shared = f"{4 * D} + {4 * D}/{chunk}: the (B,D) input block is shared by the {chunk} samples of a launch and served by L2"
    pos = {
        "bwd_layer2 (distinct x, dx written)": position(bwd_calls, "distinct_x", 12 * D, f"{12 * D} (x, dy in; dx out)"),
        "bwd_layer1 (shared x, no dx)": position(bwd_calls, "shared_x/nodx", 12 * D, shared + "; dy in, no dx"),
        "fwd_layer1 (shared x)": position(("whvi_layer_fwd_fused_f32",), ("shared_x", "shared_x/from_t2"), 8 * D,
                                          shared + " (its first transform hoisted: t2 = H(s2 x) once per launch); y out"),
        "fwd_layer2 (distinct x)": position(("whvi_layer_fwd_fused_f32",), "distinct_x", 8 * D, f"{8 * D} (x in, y out)"),
        "loss_layer3 (fwd + MNLL + bwd in one kernel)": position(("whvi_layer_loss_f32",), "distinct_x", 8 * D,
                                                                  f"{8 * D} (x in, dx out; the target is L2-resident)"),
    }
    dom = pos["bwd_layer2 (distinct x, dx written)"]
    roofline = {"bound": "hbm", "kernel": "layer_bwd_tm_kernel (+ layer_bwd_reduce_{slabs,fold}_kernel) at the layer-2 position: "
                                          "per-sample x and dy in, dx out",
                "achieved": dom["achieved"], "peak": peak, "unit": "GB/s", "frac": dom["frac"],
                "frac_of_8TBs_nominal": dom["frac_of_8TBs_nominal"], "traffic": None,
                "traffic_note": "not measured in-run (needs ncu); profiles/r02_ncu_*.txt holds dram__bytes of the same kernel and shape",
                "algorithmic_bytes_per_launch": 12.0 * D * rows_per_launch, "peak_source": peak_src,
                "algorithmic_bytes_per_row": 12 * D, "rows_per_launch": rows_per_launch, "avg_launch_ms": dom["avg_launch_ms"],
                "launches_timed": dom["launches_timed"], "share_of_step": dom["share_of_step"], "positions": pos}
    lk = pos["loss_layer3 (fwd + MNLL + bwd in one kernel)"]
    if lk:
        roofline["loss_kernel"] = dict(lk, kernel="layer_loss_tm_kernel (+ reductions)",
                                       note="replaces a forward (8 B/elt) + backward (12 B/elt) pair of the last layer")
    f2 = pos["fwd_layer2 (distinct x)"]
    if f2:
        roofline["fwd_kernel"] = dict(f2, kernel="layer_fwd_kernel at the layer-2 position")
    # whole step against the same roofline: SURVEY 8d's 20*D bytes per (sample, row, layer) over all ranks
    step_bytes = 20.0 * D * S_TOTAL * B * N_LAYERS
    step_gbs = step_bytes / (ms_step * 1e-3) / 1e9
    roofline["whole_step"] = {"algorithmic_bytes_per_step": step_bytes, "achieved": step_gbs, "unit": "GB/s",
                              "frac": step_gbs / (peak * world), "n_gpus": world,
                              "note": "SURVEY 8d yardstick: fwd 8*D + bwd 12*D bytes per (sample, row, layer); the fused last layer, "
                                      "the shared first-layer input and the skipped first-layer dx move fewer bytes than this"}

    # ---- FWHT GB/s sweep (second half of BASELINE.json's metric) on every rank: rows sharded, no collective; 2^28
    # elements = 1 GiB in + 1 GiB out per rank; aggregate = N x bytes / max-over-ranks time
    n = 1 << 28
    xf, yf = torch.randn(n, device=dev), torch.empty(n, device=dev)
    fw = []
    for k in range(6, 16):
        Dk = 1 << k
        xv, yv = xf.view(n // Dk, Dk), yf.view(n // Dk, Dk)
        for _ in range(3):
            fwht_(xv, out=yv)
        ms = timed(lambda: fwht_(xv, out=yv), 10)
        gbs = world * 8.0 * n * 10 / (ms * 1e-3) / 1e9
        fw.append({"D": Dk, "gbs": round(gbs, 1), "frac_of_measured": round(gbs / (peak * world), 4),
                   "frac_of_8TBs_nominal": round(gbs / (8000.0 * world), 4)})
    # the same sweep with bf16 activations in HBM (SURVEY 8f N4; fp32 butterflies, one rounding at the store): 4 B/element
    xb, yb = xf.to(torch.bfloat16), torch.empty(n, device=dev, dtype=torch.bfloat16)
    fw16 = []
    for k in (6, 8, 10, 12, 13, 15):
        Dk = 1 << k
        xv, yv = xb.view(n // Dk, Dk), yb.view(n // Dk, Dk)
        for _ in range(3):
            fwht_(xv, out=yv)
        ms = timed(lambda: fwht_(xv, out=yv), 10)
        gbs = world * 4.0 * n * 10 / (ms * 1e-3) / 1e9
        fw16.append({"D": Dk, "gbs": round(gbs, 1), "frac_of_measured": round(gbs / (peak * world), 4),
                     "elements_per_s_vs_f32": round((gbs / 4.0) / (fw[k - 6]["gbs"] / 8.0), 3)})
    del xf, yf, xb, yb

    # ---- MC predictive evaluation (BASELINE config 5) over all ranks
    ev = None
    if not args.no_eval:
        from tools.bench_eval import run_eval
        ev = run_eval(dev, rank, world, inputs=args.eval_inputs)

    out = None
    if rank == 0:
        cpu = cpu_f = gpu_f = None
        if world == 1 and not args.no_cpu_baseline:  # CPU legs at N = 1 only: no other ranks spinning on the host cores
            cpu = cpu_layer_baseline()
            cpu_f = cpu_fwht_baseline()
            gpu_f = gpu_fwht_reference_baseline(fwht_, dev)
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": dict(CONFIG, rows_counted="S*B*layers per step", parallelism=f"mc-sample-shard x{world}",
                              samples_per_launch=chunk,
                              l2=f"inputs larger than L2 ({chunk * B * D * 4 / 2**30:.0f} GiB activations per launch)",
                              step="fwd + MNLL + KL + bwd + flat grad all-reduce (N>1) + fused Adam",
                              fusion="ReLU folded into the layer kernels; last layer fwd+MNLL+bwd in one kernel"),
               "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e,
                       "h2d_bytes_per_step": int(x_host.numel() * 4 + y_host.numel() * 4), "d2h_bytes_per_step": 4,
                       "last_loss": e2e_losses[-1]},
               "check": check, "host_enqueue_ms_per_step": host_enqueue_ms, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
               "fwht": {"elements_per_gpu": n, "unit": "GB/s", "n_gpus": world, "scaling": "weak (rows sharded, no collective)",
                        "sweep": fw, "bf16_io_sweep": fw16, "cpu_baseline": cpu_f, "ref_cuda_baseline": gpu_f},
               "eval": ev, "clocks": clk.summary()}
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=32, help="MC samples per kernel launch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eval", action="store_true")
    ap.add_argument("--eval-inputs", type=int, default=0, help="inputs of the config-5 evaluation leg (0: a bounded default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the last timed step's loss, gradient and updated parameters to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the timed steps of --impl ours")
    if args.impl == "reference":
        return run_reference_arm(args)
    if int(os.environ.get("WORLD_SIZE", "1")) == 1:
        use_all_host_threads()  # the CPU-baseline legs of a single-process run use every host core
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
