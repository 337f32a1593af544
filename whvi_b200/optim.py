"""Flat parameter / gradient storage and a fused Adam step for the reference's training loop
(``src/networks.py:71-99``; the reference builds ``torch.optim.Adam`` in ``src/evaluation.py:15-27``).

A WHVI model has many small parameter vectors (4 per square block + the likelihood's sigma: 13 tensors for
the 3 x 4096 bench model, ~50 for a UCI MLP with a stacked first layer).  Per step, eager PyTorch issues a
handful of kernels PER TENSOR for the optimizer and -- multi-GPU -- a copy in and out of a communication
bucket per tensor.  Here

* ``FlatParams`` re-homes every parameter as a view into ONE contiguous fp32 buffer and every ``.grad`` as a
  view into a second one (autograd accumulates into existing ``.grad`` tensors in place, so the views
  persist): ``zero_grad`` is one memset, the multi-GPU gradient exchange is ONE NCCL all-reduce on the flat
  gradient buffer with no pack / unpack kernels;
* ``FlatAdam`` is a ``torch.optim.Optimizer`` whose ``step`` is ONE kernel (``whvi_adam_f32``) over the flat
  buffers, in ``torch.optim.Adam``'s arithmetic (tested against it); step count and (optionally) the learning
  rate live on the device, so it is CUDA-graph safe and follows ``LambdaLR`` & co. when ``lr`` is a CUDA tensor.
"""
from __future__ import annotations

from typing import Iterable, List

import torch

from . import _lib
from . import functional as WF


class FlatParams:
    """``flat = FlatParams(model.parameters())``: ``flat.param`` / ``flat.grad`` are the contiguous buffers,
    every ``p.data`` / ``p.grad`` a view into them (same values, same shapes, same ``state_dict``)."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("FlatParams needs at least one parameter that requires grad")
        dev = self.params[0].device
        for p in self.params:
            if p.dtype != torch.float32 or p.device != dev:
                raise RuntimeError("FlatParams: all parameters must be float32 on one device")
        # every segment starts on a 16-byte boundary (the layer kernels read parameters as float4)
        self.offsets, off = [], 0
        for p in self.params:
            self.offsets.append(off)
            off += (p.numel() + 3) // 4 * 4
        self.numel = off
        self.param = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(self.numel, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, o in zip(self.params, self.offsets):
                n = p.numel()
                self.param[o:o + n].copy_(p.detach().reshape(-1))
                p.data = self.param[o:o + n].view(p.shape)
                p.grad = self.grad[o:o + n].view(p.shape)

    def attached(self) -> bool:
        """True while every ``.grad`` still is this object's view (``zero_grad(set_to_none=True)`` or an
        optimizer that replaces ``.grad`` detaches them)."""
        return all(p.grad is not None and p.grad.data_ptr() == self.grad.data_ptr() + 4 * o
                   for p, o in zip(self.params, self.offsets))

    def reattach(self) -> None:
        for p, o in zip(self.params, self.offsets):
            view = self.grad[o:o + p.numel()].view(p.shape)
            if p.grad is None:
                view.zero_()
            elif p.grad.data_ptr() != view.data_ptr():
                view.copy_(p.grad)
            p.grad = view

    def zero_grad(self) -> None:
        """One memset; the ``.grad`` views stay in place (never ``set_to_none``)."""
        if not self.attached():
            self.reattach()
        self.grad.zero_()

    def all_reduce(self, group=None) -> None:
        """Sum the gradients over the ranks: one collective on the flat buffer, zero copy kernels."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        if not self.attached():
            self.reattach()
        dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=group)


class FlatAdam(torch.optim.Optimizer):
    """Adam (no weight decay, no amsgrad -- what the reference uses) as one fused kernel over ``FlatParams``.

    ``lr`` may be a float or a 0-d / 1-element CUDA tensor (then schedulers update it in place and captured
    CUDA graphs see the new value).  ``zero_grad`` is the flat memset regardless of ``set_to_none``."""

    whvi_graph_safe = True  # graphs._check_optimizer: no host-side state changes per step

    def __init__(self, flat: FlatParams, lr=1e-3, betas=(0.9, 0.999), eps=1e-8):
        if not isinstance(flat, FlatParams):
            flat = FlatParams(flat)
        self.flat = flat
        super().__init__(flat.params, dict(lr=lr, betas=betas, eps=eps))
        dev = flat.param.device
        self.exp_avg = torch.zeros_like(flat.param)
        self.exp_avg_sq = torch.zeros_like(flat.param)
        self.step_t = torch.zeros(1, dtype=torch.float32, device=dev)
        # visible as ordinary optimizer state (state_dict / checkpointing, graphs.GraphedTrainStep's save-and-restore)
        self.state[flat.params[0]] = {"step": self.step_t, "exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq}

    @torch.no_grad()
    def step(self, closure=None, grad_scale: float = 1.0):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        flat = self.flat
        if not flat.attached():
            flat.reattach()
        group = self.param_groups[0]
        lr, (b1, b2) = group["lr"], group["betas"]
        lr_dev = None
        if torch.is_tensor(lr):
            if lr.is_cuda:
                lr_dev, lr = lr, 0.0
            else:
                lr = float(lr)
        self.step_t.add_(1.0)
        dev = flat.param.device
        with torch.cuda.device(dev), WF._Timed("whvi_adam_f32"):
            rc = _lib.lib().whvi_adam_f32(flat.param.data_ptr(), flat.grad.data_ptr(), self.exp_avg.data_ptr(),
                                          self.exp_avg_sq.data_ptr(), flat.numel, float(lr),
                                          None if lr_dev is None else lr_dev.data_ptr(), self.step_t.data_ptr(),
                                          float(b1), float(b2), float(group["eps"]), float(grad_scale),
                                          torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "whvi_adam_f32")
        return loss

    def load_state_dict(self, state_dict) -> None:
        """``torch.optim.Optimizer.load_state_dict``, then the loaded step count and moments copied into the buffers the kernel
        reads, which stay this optimizer's state.  A tensor ``lr`` receives the loaded value in place and stays in the
        param group.  Everything is copied in place, so a ``graphs.GraphedTrainStep`` captured before the load stays valid."""
        groups = state_dict["param_groups"]
        pid = groups[0]["params"][0] if len(groups) == 1 and groups[0]["params"] else None
        saved = state_dict["state"].get(pid, {})
        n = self.flat.numel
        for key, size in (("step", 1), ("exp_avg", n), ("exp_avg_sq", n)):
            got = saved.get(key)
            if got is None or torch.as_tensor(got).numel() != size:
                have = "missing" if got is None else f"{torch.as_tensor(got).numel()} elements"
                raise ValueError(f"FlatAdam.load_state_dict: state '{key}' must have {size} elements "
                                 f"(this optimizer's flat buffer), got {have}")
        lr = self.param_groups[0]["lr"]
        super().load_state_dict(state_dict)
        loaded = self.state[self.flat.params[0]]
        with torch.no_grad():
            self.step_t.copy_(torch.as_tensor(loaded["step"]).reshape(1))
            self.exp_avg.copy_(loaded["exp_avg"].reshape(-1))
            self.exp_avg_sq.copy_(loaded["exp_avg_sq"].reshape(-1))
            if torch.is_tensor(lr):
                lr.copy_(torch.as_tensor(self.param_groups[0]["lr"]).reshape(lr.shape))
                self.param_groups[0]["lr"] = lr
        self.state[self.flat.params[0]] = {"step": self.step_t, "exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq}

    def zero_grad(self, set_to_none: bool = False) -> None:  # noqa: ARG002 -- the views must survive
        self.flat.zero_grad()
