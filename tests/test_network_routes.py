"""WHVI networks against an fp64 dense-weight network on every route the fused training and evaluation paths take.

``WHVINetwork._run``, ``loss``, ``predictive_sums`` and the autograd functions under them decide, for each pair of neighbouring
modules, which kernels run, and they hand flags from one autograd node to another that only work in matching pairs: a ReLU
folded into the producer's store (``relu_out``) and its mask applied in the consumer's backward (``relu_in``); the fused loss
layer's dx for a unit coefficient and the coefficient left in a ``DeferredScale`` for the producer's scaled backward.  If one
side of a pair is set wrong, the network does not crash: it computes the gradient of a slightly different function.

This file restates those routing rules as small predicates, each citing the source line it rests on (CPU, with the cited
lines checked, and the predicates checked against the library's own on a grid of modules).  It lists the route cells, gives
every cell a network and checks that each cell's network takes that route.  On the GPU every cell runs with injected noise
and is compared, tensor by tensor, with an fp64 network rebuilt from the same parameters and noise: the loss, every
parameter gradient and dx, in the norm max|a - b| / max|b| (``rel_err``).  Launch counts and the autograd graph confirm each
cell took its route (below): a cell that passes on the wrong route does not count as covered.

The fp64 network.  A square block is W_s = diag(s1) H diag(g_s) H diag(s2) with g_s = mu + softplus(rho) eps_s (or mu + L eps_s
for the dense posterior); it is applied as s1 * H(g_s * H(s2 * x)) with an fp64 torch FWHT (``fwht64``), which a CPU test ties
to the dense W_s, to ``O.paper_weight`` and to the pinned ``tests/golden/paper.npz``.  A Stacked layer zero-pads its input to
D_in, stacks its blocks and truncates to n_out; a Column layer takes row 0 of its block; a ``WHVIConv2d`` is ``F.conv2d`` with
the dense blocks' filters; ``semantics="reference"`` is the map the reference executes, D diag(s1 g s2) (tied to
``O.ref_sample_lrt``).  The losses are the Gaussian MNLL from the likelihood's formula (tied to ``tests/golden/mnll.npz``) or the
fp64 ``log_softmax`` NLL, plus the KL (tied to the oracle and ``tests/golden/kl.npz``).

Tolerances.  fp32: 1e-4 per tensor, DESIGN §2's bound for layers; every fp32 cell stays within it (the largest error measured
on one B200 at a 1000 W power limit is 1.5e-6).  bf16: the same fp64 network on the bf16-rounded input.  Each WHVI layer rounds
its activation and its dx once (2^-8 relative each), but the g_rho / g_mu gradients are sums over the samples of terms of
either sign, which cancel, so the relative error of the sum is not bounded by the roundings alone.  The bound is therefore
empirical: 8 * 2^-8 per WHVI layer (``_bf16_tol``), the largest measured errors plus headroom.  Measured: 4.4e-2 for the padded
D = 2 network's g_rho (bound 6.3e-2) and 5.5e-2 for the three-layer holder network's first-layer g_rho (bound 9.4e-2); every
other bf16 cell is below 1.6e-2.  A route set wrong costs far more: a ReLU mask dropped, or a loss coefficient of about 4.5
applied twice or never.  Classifier inputs are scaled so that the largest logit is about 4 (``_setup``).

Routes.  ``WF.LAUNCH_COUNTS`` shows the loss layer, the producer's scaled backward (fp32), the hoisted transform and the
multi-pass backward; the autograd graph of the loss (``observed_route``) shows the ReLUs left unfolded, the layers whose
backward applies a folded ReLU's mask, the holder (fp32 and bf16), forward_sqerr and the categorical NLL.  Both are checked
against the restated route of every training cell.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from pathlib import Path
from typing import Callable

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import rel_err
from oracle import oracle as O

PKG = Path(__file__).resolve().parent.parent / "whvi_b200"
TOL = 1e-4
BF16_U = 2.0 ** -8


def dev():
    return torch.device("cuda:0")


# ------------------------------------------------------------------------------------------------- the routing rules, restated
MIN_LAYER_D, FUSED_BWD_MAX_D = 4, 8192            # functional.py:576, :347
LOSS_LAYER_MIN_D, LOSS_LAYER_MAX_D = 128, 4096     # functional.py:474
FUSED_MOMENTS_MIN_D, FUSED_MOMENTS_MAX_D = 8192, 32768   # functional.py:240
HOIST_MIN_ELEMENTS = 1 << 24                       # functional.py:577

CITED = [
    ("functional.py", 576, "MIN_LAYER_D = 4"),
    ("functional.py", 347, "FUSED_BWD_MAX_D = 8192"),
    ("functional.py", 474, "LOSS_LAYER_MIN_D, LOSS_LAYER_MAX_D = 128, 4096"),
    ("functional.py", 240, "FUSED_MOMENTS_MIN_D, FUSED_MOMENTS_MAX_D = 8192, 32768"),
    ("functional.py", 577, "HOIST_MIN_ELEMENTS = 1 << 24"),
    ("functional.py", 409, "if D > FUSED_BWD_MAX_D:"),
    ("functional.py", 547, "if x.dtype == torch.bfloat16:"),
    ("functional.py", 549, "elif x.dim() == 2 and g.size(0) >= 4 and g.size(-1) >= 128 and g.size(0) * x.numel() >= HOIST_MIN_ELEMENTS:"),
    ("functional.py", 568, "scale = ctx.dy_scale_from.take() if ctx.dy_scale_from is not None else None"),
    ("functional.py", 653, "ctx.dx_scale_to = dx_scale_to if (want_dx and not ctx.shared_x) else None"),
    ("functional.py", 666, "if ctx.shared_x:"),
    ("functional.py", 667, "dx = dx.sum(dim=0) * c"),
    ("functional.py", 668, "elif ctx.dx_scale_to is not None:"),
    ("functional.py", 669, "ctx.dx_scale_to.put(c.reshape(1))"),
    ("functional.py", 671, "dx = dx * c"),
    ("weights.py", 203, "if h.dtype == torch.bfloat16:"),
    ("weights.py", 204, "y = self.sample_lrt(h, bias=self.bias, relu_in=relu_in)"),
    ("weights.py", 197, 'return self.semantics == "paper" and WF.MIN_LAYER_D <= self.D <= WF.FUSED_BWD_MAX_D'),
    ("weights.py", 234, "return self.fusable and WF.LOSS_LAYER_MIN_D <= self.D <= WF.LOSS_LAYER_MAX_D"),
    ("weights.py", 293, 'return self.one_launch and w.semantics == "paper" and w.fusable'),
    ("weights.py", 296, "loss_fusable = False"),
    ("weights.py", 395, "self.loss_fusable = False"),
    ("weights.py", 429, 'return self.one_launch and sub.semantics == "paper"'),
    ("networks.py", 79, "return (isinstance(module, WHVILinear) and isinstance(module.weight_submodule, WHVISquarePow2Matrix)"),
    ("networks.py", 80, "and module.weight_submodule.fusable)"),
    ("networks.py", 85, "isinstance(module.weight_submodule, WHVIStackedMatrix) and module.weight_submodule.grouped"),
    ("networks.py", 90, "isinstance(module.weight_submodule, WHVIColumnMatrix) and module.weight_submodule.fused"),
    ("networks.py", 95, "return (cls._fusable_square(module) or cls._fusable_stacked(module)"),
    ("networks.py", 96, "or (cls._fusable_column(module) and module.weight_submodule.transposed))"),
    ("networks.py", 120, "if self.fuse and self._fusable_stacked(module):"),
    ("networks.py", 123, "relu_out = (i + 2 < len(modules) and type(modules[i + 1]) is nn.ReLU and self._relu_fusable(modules[i + 2]))"),
    ("networks.py", 128, "if self.fuse and self._fusable_column(module):"),
    ("networks.py", 130, "relu_out = (not w.transposed and i + 2 < len(modules) and type(modules[i + 1]) is nn.ReLU"),
    ("networks.py", 136, "if self.fuse and self._fusable_square(module):"),
    ("networks.py", 138, "relu_out = (i + 2 < len(modules) and type(modules[i + 1]) is nn.ReLU"),
    ("networks.py", 140, "if last and sqerr_target is not None and w.loss_fusable and torch.is_grad_enabled():"),
    ("networks.py", 143, "sq = w.forward_loss(h, sqerr_target, relu_in=relu_in, dx_scale_to=scale_holder)"),
    ("networks.py", 145, "elif last and sqerr_target is not None:"),
    ("networks.py", 150, "scale_holder = (WF.DeferredScale() if (relu_out and i + 2 == len(modules) - 1 and sqerr_target is not None"),
    ("networks.py", 151, "and nxt.loss_fusable and torch.is_grad_enabled()) else None)"),
    ("networks.py", 185, "fused = (self.fuse and isinstance(self.likelihood, GaussianLikelihood) and modules"),
    ("networks.py", 186, "and self._fusable_square(modules[-1]) and x.dim() == 2 and y.dim() == 2"),
    ("networks.py", 187, "and y.size(1) == modules[-1].weight_submodule.D and y.size(0) == x.size(0) and y.is_cuda)"),
    ("networks.py", 192, "elif isinstance(self.likelihood, CategoricalLikelihood):"),
    ("networks.py", 197, "self.current_mnll = self.likelihood.mnll_batch_estimate(y, self(x), n)"),
    ("networks.py", 246, "if not (self.fuse and modules and self._fusable_square(modules[-1]) and X.dim() == 2 and X.is_cuda):"),
    ("networks.py", 256, "if h.dim() == 2 or (h.dim() == 3 and h.stride(0) == 0):"),
    ("networks.py", 265, "if WF.FUSED_MOMENTS_MIN_D <= last.D <= WF.FUSED_MOMENTS_MAX_D:"),
    ("networks.py", 268, "WF.mc_moments_(WF.layer_forward_raw(h, g, last.s1, last.s2, bias), sum_y, sum_y2, accumulate=False)"),
    ("networks.py", 294, "if loss is _rmse_of_mc_mean and y_test.dim() == 2:"),
    ("networks.py", 297, "if sums is not None and sums[0].shape == y_test.shape:"),
    ("networks.py", 316, 'sums = None if self.rng_mode == "reference" else self.predictive_sums(X, S)'),
]


def _w(m):
    return getattr(m, "weight_submodule", None)


def square_fusable(w):
    """weights.py:197: PAPER semantics and MIN_LAYER_D <= D <= FUSED_BWD_MAX_D."""
    return w.semantics == "paper" and MIN_LAYER_D <= w.D <= FUSED_BWD_MAX_D


def square_loss_fusable(w):
    """weights.py:234: fusable and LOSS_LAYER_MIN_D <= D <= LOSS_LAYER_MAX_D."""
    return square_fusable(w) and LOSS_LAYER_MIN_D <= w.D <= LOSS_LAYER_MAX_D


def stacked_grouped(w):
    """weights.py:293: one_launch, PAPER semantics and a fusable block."""
    b = w.weight_matrices[0]
    return w.one_launch and b.semantics == "paper" and square_fusable(b)


def column_fused(w):
    """weights.py:429: one_launch and PAPER semantics."""
    return w.one_launch and w.weight_submodule.semantics == "paper"


def kind(m):
    """'square' / 'stacked' / 'column' for a WHVILinear by its weight module (networks.py:79, :85, :90), else None: a
    WHVIConv2d is none of them."""
    from whvi_b200 import WHVILinear
    from whvi_b200.weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix
    if not isinstance(m, WHVILinear):
        return None
    return {WHVISquarePow2Matrix: "square", WHVIStackedMatrix: "stacked", WHVIColumnMatrix: "column"}[type(m.weight_submodule)]


def fusable_square(m):
    return kind(m) == "square" and square_fusable(_w(m))       # networks.py:79-80


def fusable_stacked(m):
    return kind(m) == "stacked" and stacked_grouped(_w(m))     # networks.py:85


def fusable_column(m):
    return kind(m) == "column" and column_fused(_w(m))         # networks.py:90


def relu_fusable(m):
    """networks.py:95-96: the consumer's kernels can apply a folded ReLU's mask: a fused square or Stacked layer, or a fused
    Column layer in its n -> 1 (transposed) form."""
    return fusable_square(m) or fusable_stacked(m) or (fusable_column(m) and _w(m).transposed)


def hoists(S, B, D, shared, bf16):
    """functional.py:547-549: a shared fp32 input with S >= 4, D >= 128 and S B D >= 2^24 gets its first transform once."""
    return shared and not bf16 and S >= 4 and D >= 128 and S * B * D >= HOIST_MIN_ELEMENTS


def loss_dx_outcome(want_dx, shared_x, holder):
    """WHVILayerLossFunction (functional.py:653, :666-671): what its backward does with dx."""
    if not want_dx:
        return "none"
    if shared_x:
        return "sum_then_scale"             # :666-667
    return "holder" if holder else "scale_here"   # :653, :668-671 (scale_here: a new tensor, the saved dx stays as it is)


def gaussian_fused(modules, fuse, x_dim, y_shape, x_rows):
    """networks.py:185-187: the Gaussian data term goes through ``_run`` with a target."""
    return bool(fuse and modules and fusable_square(modules[-1]) and x_dim == 2 and len(y_shape) == 2
                and y_shape[1] == _w(modules[-1]).D and y_shape[0] == x_rows)


def restated_run(modules, *, fuse, S, B, x_dim, target, grad, bf16):
    """networks.py:115-162 for a network of ``modules``: the set of route tags one ``_run`` produces.
      fold@i        the ReLU at index i is folded into its producer (:123, :130-131, :138-139)
      unfolded@i    the ReLU at index i runs as its own module
      relu_in@i     module i's backward applies a folded ReLU's mask
      loss_layer    the last square layer is the fused loss layer (:140), with dx:<outcome> of ``loss_dx_outcome``
      holder        a producer shares a DeferredScale with the loss layer (:150-151)
      sqerr         the last square layer runs forward_sqerr (:145): WHVILayerSqErrFunction in fp32, sqerr_bf16 in bf16
      hoist         a square layer on the hoisted-t2 path (functional.py:549)
      multipass     a square layer past FUSED_BWD_MAX_D (functional.py:409)"""
    tags, n = set(), len(modules)
    i, relu_in, holder, sampled, shared = 0, False, False, False, x_dim == 2
    while i < n:
        m, last = modules[i], i == n - 1
        k = kind(m)
        whvi = k is not None or type(m).__name__ == "WHVIConv2d"
        if relu_in:
            tags.add(f"relu_in@{i}")
        if fuse and (fusable_stacked(m) or fusable_column(m)):
            relu_out = (not (k == "column" and _w(m).transposed) and i + 2 < n and type(modules[i + 1]) is nn.ReLU
                        and relu_fusable(modules[i + 2]))
            holder = False
        elif fuse and fusable_square(m):
            w = _w(m)
            relu_out = i + 2 < n and type(modules[i + 1]) is nn.ReLU and relu_fusable(modules[i + 2])
            if last and target and square_loss_fusable(w) and grad:
                tags |= {"loss_layer", "dx:" + loss_dx_outcome(True, not sampled and shared, holder)}
                if holder:
                    tags.add("holder")
            elif last and target:
                tags.add("sqerr_bf16" if bf16 else "sqerr")   # weights.py:203-205: bf16 is the layer, then a torch sum
            else:
                holder = (relu_out and i + 2 == n - 1 and target and square_loss_fusable(_w(modules[i + 2])) and grad)
                if hoists(S, B, w.D, not sampled and shared, bf16):
                    tags.add("hoist")
        else:
            relu_out = False
            if k == "square" and _w(m).semantics == "paper" and _w(m).D >= MIN_LAYER_D and hoists(S, B, _w(m).D, not sampled and shared, bf16):
                tags.add("hoist")
            if type(m) is nn.ReLU:
                tags.add(f"unfolded@{i}")
        if k == "square" and _w(m).D > FUSED_BWD_MAX_D:
            tags.add("multipass")
        if relu_out:
            tags.add(f"fold@{i + 1}")
        relu_in = relu_out
        sampled = sampled or whvi
        i += 2 if relu_out else 1
    return tags


def restated_loss(net, x_shape, y_shape, grad, bf16=False):
    """networks.py:185-197: the route of ``net.loss`` -- the fused Gaussian path through ``_run``, the categorical NLL on the
    (S, B, K) logits, or torch's ``mnll_batch_estimate`` on ``forward()`` -- with ``restated_run``'s tags."""
    from whvi_b200.likelihoods import CategoricalLikelihood
    modules = list(net.sequential.children())
    S = net.train_samples if net.training else net.eval_samples
    fused = isinstance(net.likelihood, nn.Module) and not isinstance(net.likelihood, CategoricalLikelihood) and \
        gaussian_fused(modules, net.fuse, len(x_shape), y_shape, x_shape[0])
    tags = restated_run(modules, fuse=net.fuse, S=S, B=x_shape[0], x_dim=len(x_shape), target=fused, grad=grad, bf16=bf16)
    if isinstance(net.likelihood, CategoricalLikelihood):
        tags.add("categorical")
    elif not fused:
        tags.add("torch_mnll")
    return tags


def observed_route(loss):
    """The route as the autograd graph of ``loss`` records it: the ReLUs that run as their own op (``ReluBackward0``), the
    layers whose backward applies a folded ReLU's mask (``relu_in`` on the ctx of WHVILayerFunction and WHVILayerSqErrFunction,
    in ``meta`` of the Stacked and Column functions), producers that share a DeferredScale (``dy_scale_from``), the fused loss
    layer, forward_sqerr's function and the categorical NLL.  The loss layer does not keep its relu_in, so it is not counted."""
    out = dict.fromkeys(("relu", "relu_in", "holder", "loss_layer", "sqerr", "categorical"), 0)
    seen, stack = set(), [loss.grad_fn]
    while stack:
        node = stack.pop()
        if node is None or node in seen:
            continue
        seen.add(node)
        name = type(node).__name__
        if name == "ReluBackward0":
            out["relu"] += 1
        elif name == "WHVILayerFunctionBackward":
            out["relu_in"] += bool(node.relu_in)
            out["holder"] += node.dy_scale_from is not None
        elif name == "WHVILayerSqErrFunctionBackward":
            out["sqerr"] += 1
            out["relu_in"] += bool(node.relu_in)
        elif name in ("WHVIStackedFunctionBackward", "WHVIStackedGFunctionBackward"):
            out["relu_in"] += bool(node.meta[8])     # (S, B, D, G, xs, n_in, n_out, stride, relu_in, ...)
        elif name in ("WHVIColumnFunctionBackward", "WHVIColumnGFunctionBackward"):
            out["relu_in"] += bool(node.meta[6])     # (S, B, D, n, xs, transposed, relu_in, has_bias)
        elif name == "WHVILayerLossFunctionBackward":
            out["loss_layer"] += 1
        elif name == "CategoricalNLLFunctionBackward":
            out["categorical"] += 1
        stack.extend(f for f, _ in node.next_functions)
    return out


def expected_route(tags, n_modules):
    """``observed_route`` as the restated tags predict it."""
    loss_idx = n_modules - 1 if "loss_layer" in tags else None
    return {"relu": sum(t.startswith("unfolded@") for t in tags),
            "relu_in": sum(t.startswith("relu_in@") and int(t[8:]) != loss_idx for t in tags),
            "holder": int("holder" in tags), "loss_layer": int("loss_layer" in tags), "sqerr": int("sqerr" in tags),
            "categorical": int("categorical" in tags)}


def restated_sums(net, X_dim):
    """networks.py:246-268: the route of ``predictive_sums``: None (no sums), 'predictive_moments' (no WHVI layer before the
    last, :256), 'moments' (the fused moments kernel, :265) or 'mc_moments' (a forward, then ``mc_moments_``, :268)."""
    modules = list(net.sequential.children())
    if not (net.fuse and modules and fusable_square(modules[-1]) and X_dim == 2):
        return None
    if not any(kind(m) is not None or type(m).__name__ == "WHVIConv2d" for m in modules[:-1]):
        return "predictive_moments"
    D = _w(modules[-1]).D
    return "moments" if FUSED_MOMENTS_MIN_D <= D <= FUSED_MOMENTS_MAX_D else "mc_moments"


def key_calls(tags, bf16, backward=True):
    """The C-ABI calls that tell the routes apart, per loss forward (+ backward): the loss layer, the producer's scaled
    backward, the hoisted transform."""
    loss = "whvi_layer_loss_bf16" if bf16 else "whvi_layer_loss_f32"
    return {loss: int("loss_layer" in tags), "whvi_layer_bwd_scaled_f32": int("holder" in tags and backward and not bf16),
            "whvi_fwht_scaled_f32": int("hoist" in tags)}


def sums_calls(route, D, S, chunk=16):
    if route == "moments":
        return {"whvi_layer_moments_f32": 1, "whvi_mc_moments_f32": 0, "whvi_fwht_scaled_f32": 0}
    if route == "mc_moments":
        return {"whvi_layer_moments_f32": 0, "whvi_mc_moments_f32": 1, "whvi_fwht_scaled_f32": 0}
    fused = FUSED_MOMENTS_MIN_D <= D <= FUSED_MOMENTS_MAX_D   # functional.py:327
    return {"whvi_layer_moments_f32": int(fused), "whvi_mc_moments_f32": 0 if fused else -(-S // chunk), "whvi_fwht_scaled_f32": 1}


# ------------------------------------------------------------------------------------------------- networks and cells
def L(*a, **k):
    from whvi_b200 import WHVILinear
    return WHVILinear(*a, lambda_=2.0, **k)


def Conv(*a, **k):
    from whvi_b200 import WHVIConv2d
    return WHVIConv2d(*a, lambda_=2.0, **k)


@dataclass
class Net:
    modules: Callable[[], list]
    x: tuple                  # input shape
    S: int = 3
    out: int = 0              # Gaussian targets (B, out); 0: a classifier
    K: int = 0                # classes
    xgrad: bool = True
    n: int = 1000             # data-set size of the loss (!= B)
    eval_S: int = 3
    chunk: int | None = None


NETS = {
    # the Gaussian loss, fused loss layer
    "holder": Net(lambda: [L(8, 128, bias=True), nn.ReLU(), L(128, 128, bias=True), nn.ReLU(), L(128, 128, bias=True)],
                  (33, 8), out=128),
    "holder_dense": Net(lambda: [L(8, 128, bias=True, covariance="dense"), nn.ReLU(), L(128, 128, covariance="dense"), nn.ReLU(),
                                 L(128, 128, bias=True, covariance="dense")], (17, 8), out=128),
    "square_no_relu": Net(lambda: [L(8, 256, bias=True), nn.ReLU(), L(256, 256, bias=True), L(256, 256)], (21, 8), out=256),
    "stacked_relu_loss": Net(lambda: [L(12, 256, bias=True), nn.ReLU(), L(256, 256, bias=True)], (19, 12), out=256),
    "stacked_relu_dense": Net(lambda: [L(12, 256, bias=True, covariance="dense"), nn.ReLU(), L(256, 256, covariance="dense")],
                              (19, 12), out=256),
    "column_relu_loss": Net(lambda: [L(1, 128, bias=True), nn.ReLU(), L(128, 128, bias=True)], (25, 1), out=128),
    "loss_first": Net(lambda: [L(256, 256, bias=True)], (23, 256), out=256),
    "hoist": Net(lambda: [L(4096, 4096, bias=True), nn.ReLU(), L(4096, 4096, bias=True)], (1024, 4096), S=4, out=4096),
    # the Gaussian loss, other routes
    "sqerr_64": Net(lambda: [L(4, 64, bias=True), nn.ReLU(), L(64, 64, bias=True)], (27, 4), out=64),
    "sqerr_8192": Net(lambda: [L(16, 8192, bias=True), nn.ReLU(), L(8192, 8192, bias=True)], (6, 16), S=2, out=8192),
    "multipass_16384": Net(lambda: [L(16384, 16384, bias=True), nn.ReLU(), L(16384, 16384)], (3, 16384), S=2, out=16384),
    "last_stacked": Net(lambda: [L(128, 128, bias=True), nn.ReLU(), L(128, 200, bias=True)], (15, 128), out=200),
    "last_column_t": Net(lambda: [L(64, 64, bias=True), nn.ReLU(), L(64, 1, bias=True)], (29, 64), out=1),
    "last_foreign": Net(lambda: [L(64, 64, bias=True), nn.ReLU(), nn.Linear(64, 3)], (13, 64), out=3),
    # ReLU not folded
    "relu_reference": Net(lambda: [L(64, 64, bias=True), nn.ReLU(), L(64, 64, bias=True, semantics="reference")], (11, 64), out=64),
    "relu_pad_d2": Net(lambda: [L(2, 2, bias=True), nn.ReLU(), L(2, 2, bias=True)], (31, 2), out=2),
    "relu_end": Net(lambda: [L(64, 64, bias=True), nn.ReLU()], (9, 64), out=64),
    "column_t_producer": Net(lambda: [L(64, 1, bias=True), nn.ReLU(), L(1, 64, bias=True)], (14, 64), out=64),
    # categorical loss
    "cls_square": Net(lambda: [L(12, 64, bias=True), nn.ReLU(), L(64, 64, bias=True)], (37, 12), K=64),
    "cls_stacked": Net(lambda: [L(32, 64, bias=True), nn.ReLU(), L(64, 10, bias=True)], (41, 32), K=10, eval_S=7, chunk=3),
    "cls_foreign": Net(lambda: [L(32, 32, bias=True), nn.ReLU(), nn.Linear(32, 5)], (18, 32), K=5),
    "cls_conv": Net(lambda: [Conv(2, 4, 3, padding=1, bias=True), nn.ReLU(), Conv(4, 4, 3, bias=True), nn.ReLU(), nn.Flatten(),
                             nn.Linear(64, 5)], (3, 2, 6, 6), K=5),
    # evaluation
    "sums_moments": Net(lambda: [L(8192, 8192, bias=True), nn.ReLU(), L(8192, 8192, bias=True)], (4, 8192), out=8192, eval_S=3),
    "sums_mc": Net(lambda: [L(12, 256, bias=True), nn.ReLU(), L(256, 256, bias=True)], (19, 12), out=256, eval_S=5),
    "sums_shared": Net(lambda: [nn.Linear(8, 256), nn.ReLU(), L(256, 256, bias=True)], (10, 8), out=256, eval_S=5),
}

MODES = ("train", "nograd", "scaled", "twice", "retain")
TRAIN = ["holder", "holder_dense", "square_no_relu", "stacked_relu_loss", "stacked_relu_dense", "column_relu_loss", "loss_first",
         "hoist", "sqerr_64", "sqerr_8192", "multipass_16384", "last_stacked", "last_column_t", "last_foreign", "relu_reference",
         "relu_pad_d2", "relu_end", "column_t_producer", "cls_square", "cls_stacked", "cls_foreign", "cls_conv"]
EVAL = ["forward", "sums", "eval_model", "uncertainty", "proba", "metrics"]

# (area, cell) -> (network, how it runs, route tags its restated route must contain)
CELLS = {
    ("fused loss layer", "square + ReLU producer -> holder, scaled backward"): ("holder", "train", {"loss_layer", "holder", "dx:holder", "fold@3", "relu_in@2"}),
    ("fused loss layer", "square without ReLU"): ("square_no_relu", "train", {"loss_layer", "dx:scale_here"}),
    ("fused loss layer", "Stacked + ReLU"): ("stacked_relu_loss", "train", {"loss_layer", "dx:scale_here", "fold@1", "relu_in@2"}),
    ("fused loss layer", "Column 1 -> n + ReLU (relu_in, no holder)"): ("column_relu_loss", "train", {"loss_layer", "dx:scale_here", "fold@1", "relu_in@2"}),
    ("fused loss layer", "loss layer first (shared x, dx)"): ("loss_first", "train", {"loss_layer", "dx:sum_then_scale"}),
    ("fused loss layer", "hoisted-t2 producer + ReLU + holder"): ("hoist", "train", {"loss_layer", "holder", "hoist", "fold@1"}),
    ("fused loss layer", "D = 128"): ("holder", "train", {"loss_layer"}),
    ("fused loss layer", "D = 4096"): ("hoist", "train", {"loss_layer"}),
    ("other Gaussian", "last square D = 64: forward_sqerr"): ("sqerr_64", "train", {"sqerr", "fold@1", "relu_in@2"}),
    ("other Gaussian", "last square D = 8192: forward_sqerr"): ("sqerr_8192", "train", {"sqerr", "fold@1", "relu_in@2"}),
    ("other Gaussian", "D = 16384: multi-pass backward, torch MNLL"): ("multipass_16384", "train", {"torch_mnll", "multipass", "unfolded@1"}),
    ("other Gaussian", "last Stacked with truncation"): ("last_stacked", "train", {"torch_mnll", "fold@1", "relu_in@2"}),
    ("other Gaussian", "last Column n -> 1 with relu_in"): ("last_column_t", "train", {"torch_mnll", "fold@1", "relu_in@2"}),
    ("other Gaussian", "last foreign nn.Linear"): ("last_foreign", "train", {"torch_mnll", "unfolded@1"}),
    ("other Gaussian", "loss() under torch.no_grad()"): ("holder", "nograd", {"sqerr"}),
    ("ReLU not folded", "before a foreign module"): ("last_foreign", "train", {"unfolded@1"}),
    ("ReLU not folded", "before a WHVIConv2d"): ("cls_conv", "train", {"unfolded@1", "unfolded@3"}),
    ("ReLU not folded", 'before a semantics="reference" square'): ("relu_reference", "train", {"unfolded@1", "torch_mnll"}),
    ("ReLU not folded", "before a D = 2 padded square"): ("relu_pad_d2", "train", {"unfolded@1"}),
    ("ReLU not folded", "at the end of the network"): ("relu_end", "train", {"unfolded@1", "torch_mnll"}),
    ("ReLU not folded", "Column n -> 1 as producer"): ("column_t_producer", "train", {"unfolded@1"}),
    ("coefficient", "constant != 1 and n != B, holder"): ("holder", "scaled", {"holder"}),
    ("coefficient", "constant != 1 and n != B, scaled in the loss layer"): ("square_no_relu", "scaled", {"dx:scale_here"}),
    ("coefficient", "constant != 1 and n != B, shared x"): ("loss_first", "scaled", {"dx:sum_then_scale"}),
    ("coefficient", "two backward passes into .grad, holder"): ("holder", "twice", {"holder"}),
    ("coefficient", "two backward passes into .grad, scaled in the loss layer"): ("stacked_relu_loss", "twice", {"dx:scale_here"}),
    ("coefficient", "retain_graph and a second backward, holder"): ("holder", "retain", {"holder"}),
    ("coefficient", "retain_graph and a second backward, scaled in the loss layer"): ("square_no_relu", "retain", {"dx:scale_here"}),
    ("coefficient", "retain_graph and a second backward, shared x"): ("loss_first", "retain", {"dx:sum_then_scale"}),
    ("posterior", "dense covariance, holder"): ("holder_dense", "train", {"holder"}),
    ("posterior", "dense covariance, Stacked + ReLU"): ("stacked_relu_dense", "train", {"fold@1"}),
    ("categorical", "logits from a square layer (K = D)"): ("cls_square", "train", {"categorical", "fold@1"}),
    ("categorical", "logits from a Stacked layer (K = 10)"): ("cls_stacked", "train", {"categorical", "fold@1"}),
    ("categorical", "foreign head"): ("cls_foreign", "train", {"categorical", "unfolded@1"}),
    ("categorical", "WHVIConv2d body"): ("cls_conv", "train", {"categorical"}),
    ("evaluation", "forward()"): ("holder", "forward", set()),
    ("evaluation", "predictive_sums, fused moments (D = 8192)"): ("sums_moments", "sums", {"moments"}),
    ("evaluation", "predictive_sums, mc_moments (D = 256)"): ("sums_mc", "sums", {"mc_moments"}),
    ("evaluation", "predictive_sums, no WHVI layer before the last (stride-0 expand)"): ("sums_shared", "sums", {"predictive_moments"}),
    ("evaluation", "predictive_sums with a bf16 head"): ("sums_mc", "sums_bf16", {"mc_moments"}),
    ("evaluation", "eval_model of a regressor"): ("sums_mc", "eval_model", {"mc_moments"}),
    ("evaluation", "predictive_uncertainty of a regressor"): ("sums_moments", "uncertainty", {"moments"}),
    ("evaluation", "predict_proba, S not a multiple of chunk_samples"): ("cls_stacked", "proba", set()),
    ("evaluation", "predictive_metrics, S not a multiple of chunk_samples"): ("cls_stacked", "metrics", set()),
}
# "fuse=False: every training cell again" and "bf16: every cell that accepts bf16 input" are the parametrisations of
# test_training_cell_against_fp64 over TRAIN x (fuse) x (dtype).  Every training network runs in bf16 except these, whose
# bf16 call the test checks raises instead (the hoist network runs in bf16 on the plain path: the holder route again).
BF16_REJECTED = {
    "last_foreign": "its nn.Linear has fp32 weights, which reject a bf16 input",
    "cls_foreign": "its nn.Linear head has fp32 weights, which reject a bf16 input",
    "cls_conv": "its nn.Linear head has fp32 weights, which reject a bf16 input",
    "relu_reference": 'semantics="reference" raises on bf16 activations (weights.py:178-179)',
}
BF16_NETS = [k for k in TRAIN if k not in BF16_REJECTED]

UNREACHABLE = {
    ("fused loss layer", "Stacked or Column as the loss layer"): "their loss_fusable is False (weights.py:296, :395)",
    ("fused loss layer", "holder with a shared x"): "a holder needs a square producer before the loss layer, so the loss "
                                                    "layer's input carries the sample axis (networks.py:150, functional.py:653)",
    ("fused loss layer", "D = 64 or 8192 as the loss layer"): "outside [LOSS_LAYER_MIN_D, LOSS_LAYER_MAX_D] (weights.py:234): "
                                                              "forward_sqerr instead",
    ("ReLU not folded", "Column n -> 1 producing a fold"): "networks.py:130 requires the plain (1 -> n) form",
    ("ReLU folded", "into a Column 1 -> n consumer"): "its input is 1 wide, and the only WHVI producer of a 1-wide output is "
                                                      "a Column n -> 1, which cannot produce a fold",
    ("bf16", "hoisted t2"): "functional.py:547: a bf16 input never takes the hoisted path",
    **{("bf16", name): reason for name, reason in BF16_REJECTED.items()},
}


def _build(name, fuse=True, device=None):
    from whvi_b200 import WHVIClassification, WHVIRegression
    spec = NETS[name]
    torch.manual_seed(0)
    kw = dict(train_samples=spec.S, eval_samples=spec.eval_S, fuse=fuse)
    net = WHVIClassification(spec.modules(), **kw) if spec.K else WHVIRegression(spec.modules(), sigma=1.5, **kw)
    if device is not None:
        net = net.to(device)
    return net


# ------------------------------------------------------------------------------------------------- the fp64 network
def fwht64(x):
    """Unnormalised Sylvester FWHT over the last axis, in torch (fp64, differentiable)."""
    D = x.size(-1)
    shape, h = x.shape, 1
    while h < D:
        x = x.reshape(*shape[:-1], D // (2 * h), 2, h)
        x = torch.stack((x[..., 0, :] + x[..., 1, :], x[..., 0, :] - x[..., 1, :]), dim=-2)
        h *= 2
    return x.reshape(shape)


def g64(P, b, eps):
    """(S, D) fp64 g = mu + softplus(rho) eps, or mu + L eps (tril L), for square block ``b`` with noise ``eps`` (S, D)."""
    mu = P[id(b.g_mu)]
    if b.covariance == "dense":
        return mu + eps @ torch.tril(P[id(b.g_L)]).T
    return mu + F.softplus(P[id(b.g_rho)]) * eps


def block64(P, b, eps, x):
    """y[s] = s1 * H(g_s * H(s2 * x[s])) for x (B, D) shared or (S, B, D): x W_s^T with W_s = diag(s1) H diag(g_s) H diag(s2)."""
    g = g64(P, b, eps)
    t = fwht64(P[id(b.s2)] * x)
    if t.dim() == 2:
        t = t.unsqueeze(0)
    return P[id(b.s1)] * fwht64(g[:, None, :] * t)


def dense_block64(P, b, eps):
    """(S, D, D) fp64 W_s = diag(s1) H diag(g_s) H diag(s2)."""
    Hm = torch.from_numpy(O.build_H(b.D)).to(eps.device)
    g = g64(P, b, eps)
    return P[id(b.s1)][None, :, None] * torch.einsum("ij,sj,jk->sik", Hm, g, Hm) * P[id(b.s2)][None, None, :]


def _bias(P, w):
    return None if w.bias is None else P[id(w.bias)].reshape(-1)


def linear64(P, m, eps, x):
    """A WHVILinear's map in fp64; ``eps`` maps each square block to its (S, D) noise."""
    from whvi_b200.weights import WHVIColumnMatrix, WHVIStackedMatrix
    w = m.weight_submodule
    if isinstance(w, WHVIStackedMatrix):
        xp = F.pad(x, (0, w.D_in - w.n_in))
        y = torch.cat([block64(P, b, eps[id(b)], xp) for b in w.weight_matrices], dim=-1)
        if w.bias is not None:
            y = y + _bias(P, w)
        return y[..., :w.n_out]
    if isinstance(w, WHVIColumnMatrix):
        b = w.weight_submodule
        row = (P[id(b.s1)][0] * P[id(b.s2)] * fwht64(g64(P, b, eps[id(b)])))[:, :w.D]   # row 0 of W_s, (S, n)
        xs = x.unsqueeze(0) if x.dim() == 2 else x
        y = (xs * row[:, None, :]).sum(-1, keepdim=True) if w.transposed else xs * row[:, None, :]
        return y if w.bias is None else y + _bias(P, w)
    if w.semantics == "reference":   # the map the reference executes: D diag(s1 g s2) (SURVEY F1)
        g = g64(P, w, eps[id(w)])
        y = w.D * (P[id(w.s1)] * g * P[id(w.s2)])[:, None, :] * x
    else:
        y = block64(P, w, eps[id(w)], x)
    return y if w.bias is None else y + _bias(P, w)


def conv_filters64(P, conv, eps):
    """(S, C_out, C_in, kh, kw) fp64 filters: the dense blocks stacked and truncated to (C_out, C_in kh kw)."""
    W = torch.cat([dense_block64(P, b, eps[id(b)]) for b in conv.square_blocks()], dim=1)[:, :conv.out_channels, :conv.n_in]
    kh, kw = conv.kernel_size
    return W.reshape(W.size(0), conv.out_channels, kh, kw, conv.in_channels).permute(0, 1, 4, 2, 3)


def run64(net, P, eps, x, S):
    """The network in fp64: (S, B, ...) outputs, foreign modules on the samples folded into the batch, as ``_run``."""
    from whvi_b200 import WHVIConv2d, WHVILinear
    h, sampled = x, False
    for m in net.sequential.children():
        if isinstance(m, WHVILinear):
            h, sampled = linear64(P, m, eps, h), True
        elif isinstance(m, WHVIConv2d):
            filt = conv_filters64(P, m, eps)
            bias = _bias(P, m.weight_submodule)
            bias = None if bias is None else bias[:m.out_channels]
            h = torch.stack([F.conv2d(h if h.dim() == 4 else h[s], filt[s], bias, m.stride, m.padding, m.dilation)
                             for s in range(S)])
            sampled = True
        else:
            f = {nn.ReLU: F.relu, nn.Flatten: lambda t: t.flatten(1)}.get(type(m))
            if f is None:
                f = lambda t, m=m: F.linear(t, P[id(m.weight)], P[id(m.bias)])
            if sampled:
                h = f(h.reshape(-1, *h.shape[2:])).reshape(S, -1, *f(h[0][:1]).shape[1:])
            else:
                h = f(h)
    return h if sampled else h.unsqueeze(0).expand(S, *h.shape)


def gaussian_mnll64(y, yhat, sigma, n):
    """src/likelihoods.py:18-29: -n/(m S) sum_{b,i,s} log N(y[b,i] | yhat[s,b,i], sigma), yhat (S, m, n_out)."""
    S, m = yhat.size(0), yhat.size(1)
    sq = (yhat - y).square().sum()
    count = yhat.numel()
    return -n / (m * S) * (-count * (torch.log(sigma) + 0.5 * math.log(2 * math.pi)) - 0.5 * sq / sigma ** 2)


def categorical_mnll64(y, logits, n):
    S, m = logits.size(0), logits.size(1)
    return -n / (m * S) * torch.log_softmax(logits, -1).gather(-1, y.reshape(1, m, 1).expand(S, m, 1)).sum()


def kl64(P, b, lambda_):
    """KL(q(g) || N(0, lambda I)) of one square block: the reference's diagonal formula (kl_mode 0: softplus(rho) used as a
    variance, src/utils.py:49-71; kl_mode 1: its square) or the dense one with the log-determinant (``O.kl_dense``)."""
    mu = P[id(b.g_mu)]
    D = mu.numel()
    if b.covariance == "dense":
        Lm = torch.tril(P[id(b.g_L)])
        return 0.5 * (D * math.log(lambda_) - 2 * torch.log(torch.diagonal(Lm)).sum() - D + (Lm * Lm).sum() / lambda_
                      + (mu * mu).sum() / lambda_)
    v = F.softplus(P[id(b.g_rho)])
    v = v * v if b.kl_mode else v
    return 0.5 * (D * math.log(lambda_) - torch.log(v).sum() - D + v.sum() / lambda_ + (mu * mu).sum() / lambda_)


def blocks_of(net):
    return [b for layer in net._whvi_layers() for b in layer.square_blocks()]


def loss64(net, P, eps, x, y, n, S):
    out = run64(net, P, eps, x, S)
    if net.NETKIND == "cls":
        mnll = categorical_mnll64(y, out.reshape(S, x.size(0), -1), n)
    else:
        mnll = gaussian_mnll64(y, out.reshape(S, x.size(0), -1), P[id(net.likelihood.sigma)], n)
    kl = sum(kl64(P, b, b.lambda_) for b in blocks_of(net))
    return mnll + kl


# ------------------------------------------------------------------------------------------------- CPU
def test_cited_routing_rules_are_the_source():
    """Each restated rule cites a line of whvi_b200/; the line still says it."""
    for name, line, text in CITED:
        src = (PKG / name).read_text().splitlines()
        assert text in src[line - 1], f"{name}:{line} no longer reads {text!r}: {src[line - 1]!r}"
    import whvi_b200.functional as WF
    assert (WF.MIN_LAYER_D, WF.FUSED_BWD_MAX_D, WF.LOSS_LAYER_MIN_D, WF.LOSS_LAYER_MAX_D, WF.FUSED_MOMENTS_MIN_D,
            WF.FUSED_MOMENTS_MAX_D, WF.HOIST_MIN_ELEMENTS) == (MIN_LAYER_D, FUSED_BWD_MAX_D, LOSS_LAYER_MIN_D, LOSS_LAYER_MAX_D,
                                                                 FUSED_MOMENTS_MIN_D, FUSED_MOMENTS_MAX_D, HOIST_MIN_ELEMENTS)


def _module_grid():
    from whvi_b200 import WHVIConv2d, WHVILinear
    mods = [nn.ReLU(), nn.Linear(4, 4), WHVIConv2d(2, 4, 3), WHVIConv2d(1, 8, 2)]
    for cov in ("diag", "dense"):
        for sem in ("paper", "reference"):
            if cov == "dense" and sem == "reference":
                continue
            for D in (2, 4, 64, 128, 4096, 8192, 16384):
                shapes = [(D, D), (1, D), (D, 1)]
                if D <= 4096:
                    shapes += [(D, 3 * D), (D + 1, 2 * D + 3), (3, D)]
                for n_in, n_out in shapes:
                    if cov == "dense" and max(n_in, n_out) > 4096:
                        continue      # a dense (D, D) L per block: the grid keeps to what builds in a moment
                    for one_launch in (True, False):
                        m = WHVILinear(n_in, n_out, semantics=sem, covariance=cov)
                        if hasattr(m.weight_submodule, "one_launch"):
                            m.weight_submodule.one_launch = one_launch
                        elif not one_launch:
                            continue
                        mods.append(m)
    return mods


def test_restated_predicates_are_the_library():
    """_fusable_square / _fusable_stacked / _fusable_column / _relu_fusable and the modules' fusable, loss_fusable, grouped and
    fused properties against the restated predicates, for every WHVILinear shape (square, Stacked, Column both ways), both
    semantics, one_launch on and off, D = 2 ... 16384 and both posteriors."""
    from whvi_b200 import WHVINetwork
    from whvi_b200.weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix
    torch.manual_seed(0)
    seen = set()
    for m in _module_grid():
        assert WHVINetwork._fusable_square(m) == fusable_square(m)
        assert WHVINetwork._fusable_stacked(m) == fusable_stacked(m)
        assert WHVINetwork._fusable_column(m) == fusable_column(m)
        assert WHVINetwork._relu_fusable(m) == relu_fusable(m)
        w = _w(m)
        if isinstance(w, WHVISquarePow2Matrix):
            assert (w.fusable, w.loss_fusable) == (square_fusable(w), square_loss_fusable(w))
            seen.add(("square", w.D, w.fusable, w.loss_fusable))
        elif isinstance(w, WHVIStackedMatrix):
            assert w.grouped == w.fusable == stacked_grouped(w) and w.loss_fusable is False
            seen.add(("stacked", w.grouped))
        elif isinstance(w, WHVIColumnMatrix):
            assert w.fused == column_fused(w) and w.loss_fusable is False
            seen.add(("column", w.transposed, w.fused, relu_fusable(m)))
    # the grid reaches both sides of every predicate
    assert {("square", D, D >= 4, 128 <= D <= 4096) for D in (2, 4, 64, 128, 4096, 8192)} <= seen
    assert ("square", 16384, False, False) in seen
    assert {("stacked", True), ("stacked", False), ("column", True, True, True), ("column", False, True, False),
            ("column", True, False, False)} <= seen


def test_restated_dx_outcomes_and_hoist():
    assert loss_dx_outcome(False, False, True) == "none"
    assert loss_dx_outcome(True, True, True) == "sum_then_scale"
    assert loss_dx_outcome(True, False, True) == "holder"
    assert loss_dx_outcome(True, False, False) == "scale_here"
    assert hoists(4, 1024, 4096, True, False) and not hoists(4, 1023, 4096, True, False)
    assert not hoists(3, 1 << 20, 4096, True, False) and not hoists(4, 1 << 20, 64, True, False)
    assert not hoists(4, 1024, 4096, False, False) and not hoists(4, 1024, 4096, True, True)


def test_every_route_cell_is_covered():
    """Every cell has a network and a way to run it, its network's restated route contains the cell's tags, and no cell is
    both covered and listed as unreachable."""
    assert not set(CELLS) & set(UNREACHABLE)
    for cell, (name, mode, tags) in CELLS.items():
        assert name in NETS and mode in MODES + tuple(EVAL) + ("sums_bf16",), cell
        net = _build(name)
        spec = NETS[name]
        if mode in EVAL or mode == "sums_bf16":
            if tags:
                assert {restated_sums(net, len(spec.x))} == tags, (cell, restated_sums(net, len(spec.x)))
            continue
        y_shape = (spec.x[0], spec.out) if spec.out else (spec.x[0],)
        got = restated_loss(net, spec.x, y_shape, grad=mode != "nograd")
        assert tags <= got, (cell, got)
    assert set(TRAIN) <= {name for name, mode, _ in CELLS.values() if mode == "train"}
    # a network skips bf16 only for a reason that holds: a foreign nn.Linear or a semantics="reference" layer
    from whvi_b200 import WHVILinear
    for name in TRAIN:
        mods = NETS[name].modules()
        rejects = any(type(m) is nn.Linear for m in mods) or any(
            isinstance(m, WHVILinear) and any(b.semantics == "reference" for b in m.square_blocks()) for m in mods)
        assert rejects == (name in BF16_REJECTED) == (("bf16", name) in UNREACHABLE), name


def test_fwht64_and_dense_weights_are_the_oracle(golden):
    """fwht64 is H x; the dense W_s of ``dense_block64`` is O.paper_weight; the block map is x W_s^T and, on the pinned
    paper.npz layers, reproduces the golden output and (through torch autograd) every golden gradient."""
    from whvi_b200 import WHVILinear
    rng = np.random.default_rng(0)
    for D in (2, 4, 16, 128):
        a = rng.standard_normal((3, D))
        assert np.abs(fwht64(torch.from_numpy(a)).numpy() - a @ O.build_H(D).T).max() <= 1e-12 * D
    g = golden("paper")
    for i in range(3):
        x, s1, s2, mu, rho, eps, dy = (g[f"{k}_{i}"] for k in ("x", "s1", "s2", "mu", "rho", "eps", "dy"))
        D = mu.size
        torch.manual_seed(0)
        w = WHVILinear(D, D).weight_submodule
        P = {id(p): torch.from_numpy(np.ascontiguousarray(v)).requires_grad_() for p, v in
             ((w.s1, s1), (w.s2, s2), (w.g_mu, mu), (w.g_rho, rho))}
        e = torch.from_numpy(eps)
        xt = torch.from_numpy(x).requires_grad_()
        y = block64(P, w, e, xt)
        assert rel_err(y.detach().numpy(), g[f"y_{i}"]) <= 1e-12
        Wd = dense_block64(P, w, e).detach()
        gg = g64(P, w, e).detach().numpy()
        for s in range(eps.shape[0]):
            assert rel_err(Wd[s].numpy(), O.paper_weight(gg[s], s1, s2)) <= 1e-12
            assert rel_err((xt[s] @ Wd[s].T).detach().numpy(), y[s].detach().numpy()) <= 1e-12
        (y * torch.from_numpy(dy)).sum().backward()
        for got, key in ((xt.grad, "dx"), (P[id(w.s1)].grad, "ds1"), (P[id(w.s2)].grad, "ds2"), (P[id(w.g_mu)].grad, "dmu"),
                         (P[id(w.g_rho)].grad, "drho")):
            assert rel_err(got.numpy(), g[f"{key}_{i}"]) <= 1e-11, (i, key)


def test_column_reference_and_conv_maps_are_the_oracle():
    """The Column row is O.column_weight_paper; the reference-semantics square is O.ref_sample_lrt; a conv layer's fp64 output
    is the patch matrix times the dense filters."""
    from whvi_b200 import WHVIConv2d, WHVILinear
    rng = np.random.default_rng(1)
    torch.manual_seed(0)
    for n, transposed in ((20, False), (20, True), (64, True)):
        m = WHVILinear(1, n) if not transposed else WHVILinear(n, 1)
        b = m.weight_submodule.weight_submodule
        P = {id(p): torch.from_numpy(rng.standard_normal(p.shape)) for p in m.parameters()}
        e = torch.from_numpy(rng.standard_normal((2, b.D)))
        x = torch.from_numpy(rng.standard_normal((5, n if transposed else 1)))
        y = linear64(P, m, {id(b): e}, x).numpy()
        gg = g64(P, b, e).numpy()
        for s in range(2):
            row = O.column_weight_paper(gg[s], P[id(b.s1)].numpy(), P[id(b.s2)].numpy(), n)
            ref = x.numpy() @ row[:, None] if transposed else x.numpy() * row[None, :]
            assert rel_err(y[s], ref) <= 1e-12
    m = WHVILinear(16, 16, semantics="reference")
    w = m.weight_submodule
    P = {id(p): torch.from_numpy(rng.standard_normal(p.shape)) for p in m.parameters()}
    e = torch.from_numpy(rng.standard_normal((2, 16)))
    x = torch.from_numpy(rng.standard_normal((3, 16)))
    y = linear64(P, m, {id(w): e}, x).numpy()
    sig = F.softplus(P[id(w.g_rho)]).numpy()
    for s in range(2):
        ref = O.ref_sample_lrt(x.numpy(), P[id(w.g_mu)].numpy(), sig * e[s].numpy(), P[id(w.s1)].numpy(), P[id(w.s2)].numpy())
        assert rel_err(y[s], ref) <= 1e-12
    conv = WHVIConv2d(2, 4, 3, padding=1)
    P = {id(p): torch.from_numpy(rng.standard_normal(p.shape)) for p in conv.parameters()}
    eps = {id(b): torch.from_numpy(rng.standard_normal((2, b.D))) for b in conv.square_blocks()}
    filt = conv_filters64(P, conv, eps)
    x = torch.from_numpy(rng.standard_normal((3, 2, 5, 5)))
    # patch columns in the layer's order, tap (i, j) of channel c at (i kw + j) C + c, zero-padded to the block width 32
    patches = F.pad(F.unfold(x, 3, padding=1).reshape(3, 2, 9, 25).permute(0, 3, 2, 1).reshape(3, 25, 18), (0, 14))
    (blk,) = conv.square_blocks()
    Wd = dense_block64(P, blk, eps[id(blk)])[:, :4]                                    # (S, C_out, 32)
    for s in range(2):
        via = (patches @ Wd[s].T).permute(0, 2, 1).reshape(3, 4, 5, 5).numpy()
        assert rel_err(F.conv2d(x, filt[s], padding=1).numpy(), via) <= 1e-12


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("shared", [False, True], ids=["per_sample", "shared_x"])
def test_loss_layer_backward_twice_through_a_retained_graph(monkeypatch, dtype, shared):
    """WHVILayerLossFunction's backward, run twice through a retained graph without a holder, gives c * dx both times: it
    must not scale its saved dx in place (it once did, and the second backward failed).  The kernel call is replaced by
    fixed gradients, so this runs on the CPU; the GPU cells with mode "retain" check the same on the kernels."""
    import whvi_b200.functional as WF
    S, B, D = 3, 5, 8
    gen = torch.Generator().manual_seed(0)
    kernel = {k: torch.randn(shape, generator=gen) for k, shape in
              (("dx", (S, B, D)), ("dg", (S, D)), ("ds1", (D,)), ("ds2", (D,)), ("sq", ()))}

    def fake_layer_loss_raw(x, g, s1, s2, bias, target, want_dx=True, relu_in=False):
        dx = kernel["dx"].to(x.dtype).clone() if want_dx else None
        return kernel["sq"].clone(), dx, kernel["dg"].clone(), kernel["ds1"].clone(), kernel["ds2"].clone(), None

    monkeypatch.setattr(WF, "layer_loss_raw", fake_layer_loss_raw)
    x = torch.zeros((B, D) if shared else (S, B, D), dtype=dtype, requires_grad=True)
    g, s1, s2 = (torch.zeros(shape, requires_grad=True) for shape in ((S, D), (D,), (D,)))
    sq = WF.whvi_layer_loss(x, g, s1, s2, None, torch.zeros(B, D))
    c = 1.75
    (0.5 * c * sq).backward(retain_graph=True)     # d loss / d sq = c / 2, so the coefficient is c
    first = x.grad.clone()
    (0.5 * c * sq).backward()
    dx = kernel["dx"].to(dtype)
    want = dx.sum(0) * c if shared else dx * c
    assert torch.equal(first, want)
    assert torch.equal(x.grad, first + want)
    assert torch.equal(g.grad, 2 * c * kernel["dg"]) and torch.equal(s1.grad, 2 * c * kernel["ds1"])


def test_mnll_and_kl_restatements_are_the_goldens(golden):
    """The Gaussian MNLL formula reproduces the pinned reference values; the diagonal KL equals the oracle and the pinned KL,
    with the oracle's gradients; the dense KL equals O.kl_dense."""
    g = golden("mnll")
    for key, sigma, n in (("fixed", 1.0, 12), ("rand", 15.21, 116), ("multi", 0.7, 40)):
        y, yhat = torch.from_numpy(g[f"{key}_y"]).double(), torch.from_numpy(g[f"{key}_yhat"]).double()
        v = float(gaussian_mnll64(y, yhat.permute(2, 0, 1), torch.tensor(sigma, dtype=torch.float64), n))
        assert abs(v - float(g[f"{key}_mnll"])) <= 1e-5 * max(1.0, abs(v)), key
        assert abs(v - O.mnll(g[f"{key}_y"].astype(np.float64), g[f"{key}_yhat"].astype(np.float64), sigma, n)) <= 1e-9 * abs(v)
    from whvi_b200 import WHVILinear
    k = golden("kl")
    for i in range(4):
        mu, rho, lam = k[f"mu_{i}"].astype(np.float64), k[f"rho_{i}"].astype(np.float64), float(k[f"lam_{i}"])
        torch.manual_seed(0)
        b = WHVILinear(mu.size, mu.size).weight_submodule
        P = {id(b.g_mu): torch.from_numpy(mu).requires_grad_(), id(b.g_rho): torch.from_numpy(rho).requires_grad_()}
        v = kl64(P, b, lam)
        v.backward()
        v = v.item()
        assert abs(v - float(k[f"kl_{i}"])) <= 2e-5 * max(1.0, abs(v))
        ov, odmu, odrho = O.kl(mu, rho, lam, 0, grads=True)
        assert abs(v - ov) <= 1e-12 * max(1.0, abs(ov))
        assert rel_err(P[id(b.g_mu)].grad.numpy(), odmu) <= 1e-12 and rel_err(P[id(b.g_rho)].grad.numpy(), odrho) <= 1e-12
    rng = np.random.default_rng(2)
    torch.manual_seed(0)
    b = WHVILinear(16, 16, covariance="dense").weight_submodule
    mu, Lm = rng.standard_normal(16), np.tril(rng.standard_normal((16, 16))) / 16 + 0.5 * np.eye(16)
    P = {id(b.g_mu): torch.from_numpy(mu), id(b.g_L): torch.from_numpy(Lm)}
    assert abs(float(kl64(P, b, 2.0)) - O.kl_dense(mu, Lm, 2.0)) <= 1e-12 * abs(O.kl_dense(mu, Lm, 2.0))


# ------------------------------------------------------------------------------------------------- GPU
MEASURED: dict = {}   # (cell, tensor) -> error, for the record of what the bounds leave


def check(got, ref, tol, what):
    err = rel_err(got, ref)
    MEASURED[what] = (err, tol)
    assert err <= tol, f"{what}: {err:.3e} > {tol:.1e}"


def _randomise(net, seed):
    """O(1) parameters so that every term shows: s1, s2, mu, biases and foreign weights ~ N(0, 1), rho ~ -1 + 0.3 N(0, 1),
    L = tril(N(0, 1)) / D + I / 2, sigma = 1.5 (the same idea as test_conv.py's _randomise)."""
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name == "likelihood.sigma":
                p.fill_(1.5)
            elif name.endswith("g_rho"):
                p.copy_(torch.randn(p.shape, generator=gen) * 0.3 - 1.0)
            elif name.endswith("g_L"):
                D = p.size(0)
                p.copy_(torch.tril(torch.randn(p.shape, generator=gen)) / D + torch.eye(D) * 0.5)
            else:
                p.copy_(torch.randn(p.shape, generator=gen))


def _setup(name, fuse=True, seed=0):
    spec = NETS[name]
    net = _build(name, fuse, dev())
    net.NETKIND = "cls" if spec.K else "reg"
    _randomise(net, seed + 1)
    gen = torch.Generator().manual_seed(seed + 2)
    x = torch.randn(spec.x, generator=gen)
    if spec.K:
        y = torch.randint(0, spec.K, (spec.x[0],), generator=gen)
        # a classifier's input is scaled so that its largest logit is about 4.  With O(1) parameters every layer multiplies
        # its input by about D, and logits in the thousands saturate the softmax: there one bf16 rounding of a logit (|z| 2^-9
        # absolute) moves the probabilities by far more than 2^-8.
        with torch.no_grad():
            x = x * (4.0 / float(net._run(x.to(dev()), spec.S).abs().max()))
    else:
        y = torch.randn((spec.x[0], spec.out), generator=gen) * 4.0
    return net, spec, x.to(dev()), y.to(dev())


def _noise(net, S, seed):
    gen = torch.Generator().manual_seed(seed)
    return [torch.randn((S, b.D), generator=gen).to(dev()) for b in blocks_of(net)]


def _inject(net, eps):
    for b, e in zip(blocks_of(net), eps):
        b.inject_eps(e)


def _p64(net):
    return {id(p): p.detach().double().clone().requires_grad_() for p in net.parameters()}


def _calls(counts):
    import whvi_b200.functional as WF
    return {k: v // WF._LAUNCHES_PER_CALL[k] for k, v in counts.items()}


def _bf16_tol(net):
    """8 * 2^-8 per WHVI layer, an empirical bound (see the docstring)."""
    return 8 * BF16_U * len(net._whvi_layers())


COEF = 3.0


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("fuse", [True, False], ids=["fused", "unfused"])
@pytest.mark.parametrize("name,mode", sorted({(n, m) for n, m, _ in CELLS.values() if m in MODES}))
def test_training_cell_against_fp64(name, mode, fuse, dtype):
    """loss(x, y, n) and its backward against the fp64 network, tensor by tensor: the loss, every parameter gradient and dx;
    the distinguishing launches against the restated route."""
    import whvi_b200.functional as WF
    bf16 = dtype == torch.bfloat16
    net, spec, x, y = _setup(name, fuse)
    if bf16 and name in BF16_REJECTED:   # the reason UNREACHABLE gives holds: the bf16 call raises
        with pytest.raises(RuntimeError):
            net.loss(x.to(dtype), y, n=spec.n)
        return
    net.train()
    S = spec.S
    eps = _noise(net, S, 7)
    xt = x.to(dtype).requires_grad_(spec.xgrad)
    WF.LAUNCH_COUNTS.clear()
    if mode == "nograd":
        with torch.no_grad():
            _inject(net, eps)
            loss = net.loss(xt, y, n=spec.n)
    else:
        _inject(net, eps)
        loss = net.loss(xt, y, n=spec.n)
        seen = observed_route(loss)
        if mode == "scaled":
            (COEF * loss).backward()
        elif mode == "retain":
            loss.backward(retain_graph=True)
            loss.backward()
        else:
            loss.backward()
        if mode == "twice":
            _inject(net, eps)
            loss = net.loss(xt, y, n=spec.n)
            loss.backward()
    calls = _calls(WF.LAUNCH_COUNTS)
    y_shape = tuple(y.shape)
    tags = restated_loss(net, tuple(x.shape), y_shape, grad=mode != "nograd", bf16=bf16)
    per_pass = {"twice": 2}.get(mode, 1)
    want = {k: v * per_pass for k, v in key_calls(tags, bf16, backward=mode != "nograd").items()}
    if mode == "retain":
        want["whvi_layer_bwd_scaled_f32"] *= 2
    assert {k: calls.get(k, 0) for k in want} == want, (tags, calls)
    if mode != "nograd":   # under no_grad there is no graph; the loss layer's launch count above tells sqerr from it
        assert seen == expected_route(tags, len(net.sequential)), (tags, seen)
    if "multipass" in tags:   # every layer's backward on the batched FWHT, none on the fused backward kernels
        assert calls.get("whvi_fwht_f32", 0) > 0, calls
        assert not any(calls.get(k, 0) for k in ("whvi_layer_bwd_fused_f32", "whvi_layer_bwd_scaled_f32", "whvi_layer_bwd_bf16")), calls

    P = _p64(net)
    x64 = xt.detach().double().requires_grad_(spec.xgrad)
    e64 = {id(b): e.double() for b, e in zip(blocks_of(net), eps)}
    ref = loss64(net, P, e64, x64, y.double() if not spec.K else y, spec.n, S)
    tol = _bf16_tol(net) if bf16 else TOL
    cell = f"{name}/{mode}/{'fused' if fuse else 'unfused'}/{'bf16' if bf16 else 'f32'}"
    check(loss.detach().double().cpu().numpy(), ref.detach().cpu().numpy(), tol, f"{cell}: loss")
    if mode == "nograd":
        return
    factor = {"scaled": COEF, "twice": 2.0, "retain": 2.0}.get(mode, 1.0)
    (factor * ref).backward()
    for pname, p in net.named_parameters():
        assert p.grad is not None, f"{cell}: {pname} has no gradient"
        check(p.grad.double().cpu().numpy(), P[id(p)].grad.cpu().numpy(), tol, f"{cell}: d{pname}")
    if spec.xgrad:
        check(xt.grad.double().cpu().numpy(), x64.grad.cpu().numpy(), tol, f"{cell}: dx")


def _preds64(net, spec, x, eps, S):
    P = _p64(net)
    e64 = {id(b): e.double() for b, e in zip(blocks_of(net), eps)}
    with torch.no_grad():
        return run64(net, P, e64, x.double(), S).reshape(S, x.size(0), -1)


@pytest.mark.gpu
@pytest.mark.parametrize("name,mode", sorted({(n, m) for n, m, _ in CELLS.values() if m not in MODES}))
def test_evaluation_cell_against_fp64(name, mode):
    """forward(), predictive_sums, eval_model, predictive_uncertainty, predict_proba and predictive_metrics against the same
    fp64 network's S predictions, with the distinguishing launches."""
    import whvi_b200.functional as WF
    net, spec, x, y = _setup(name, True, seed=3)
    net.eval()
    S = spec.eval_S
    cell = f"{name}/{mode}"
    if mode in ("proba", "metrics"):
        chunk = spec.chunk
        assert S % chunk != 0
        chunks = [(s0, min(S, s0 + chunk)) for s0 in range(0, S, chunk)]
        eps_c = [_noise(net, s1 - s0, 20 + i) for i, (s0, s1) in enumerate(chunks)]
        for e in eps_c:
            _inject(net, e)
        eps = [torch.cat([e[k] for e in eps_c]) for k in range(len(blocks_of(net)))]
        logits = _preds64(net, spec, x, eps, S)
        lp = torch.log_softmax(logits, -1)
        probs = lp.exp().mean(0)
        if mode == "proba":
            got = net.predict_proba(x, n_samples=S, chunk_samples=chunk)
            check(got.double().cpu().numpy(), probs.cpu().numpy(), TOL, f"{cell}: probs")
            return
        got = net.predictive_metrics(x, y, n_samples=S, chunk_samples=chunk)
        lpy = lp.gather(-1, y.reshape(1, -1, 1).expand(S, -1, 1)).squeeze(-1)     # (S, B)
        ref = {"nll": float(-(torch.logsumexp(lpy, 0) - math.log(S)).mean()), "mnll": float(-lpy.sum() / S),
               "error": float((probs.argmax(1) != y).double().mean())}
        assert got["error"] == ref["error"]
        for k in ("nll", "mnll"):
            check(np.array(got[k]), np.array(ref[k]), TOL, f"{cell}: {k}")
        return
    eps = _noise(net, S, 11)
    preds = _preds64(net, spec, x, eps, S)      # (S, B, out)
    _inject(net, eps)
    WF.LAUNCH_COUNTS.clear()
    if mode == "forward":
        got = net(x)
        check(got.detach().permute(2, 0, 1).double().cpu().numpy(), preds.cpu().numpy(), TOL, f"{cell}: predictions")
        return
    xin = x.to(torch.bfloat16) if mode == "sums_bf16" else x
    if mode == "sums_bf16":   # the head runs in bf16: the reference takes the bf16 input, the bound the head's boundaries
        preds = _preds64(net, spec, xin.float(), eps, S)
    route = restated_sums(net, xin.dim())
    D = _w(list(net.sequential.children())[-1]).D
    tol = _bf16_tol(net) if mode == "sums_bf16" else TOL
    ref_sy, ref_sy2 = preds.sum(0).cpu().numpy(), preds.square().sum(0).cpu().numpy()
    if mode in ("sums", "sums_bf16"):
        sum_y, sum_y2, S_got = net.predictive_sums(xin, S)
        assert S_got == S
        check(sum_y.double().cpu().numpy(), ref_sy, tol, f"{cell}: sum_y")
        check(sum_y2.double().cpu().numpy(), ref_sy2, tol, f"{cell}: sum_y2")
    elif mode == "eval_model":
        rmse, mnll = net.eval_model(x, y)
        mean = preds.mean(0)
        ref_rmse = float(torch.sqrt(((mean - y.double()) ** 2).mean()))
        ref_mnll = float(gaussian_mnll64(y.double(), preds, net.likelihood.sigma.detach().double(), x.size(0)))
        check(np.array(rmse), np.array(ref_rmse), TOL, f"{cell}: rmse")
        check(np.array(mnll), np.array(ref_mnll), TOL, f"{cell}: mnll")
    else:
        u = net.predictive_uncertainty(x, S)
        assert u.S == S
        check(u.mean.cpu().numpy(), preds.mean(0).cpu().numpy(), TOL, f"{cell}: mean")
        # the variance from the sums is sum_y2 / S - mean^2: fp32 sums cancel, so it is bounded relative to the second moment
        err = float((u.epistemic_variance - preds.var(0, unbiased=False)).abs().max() / preds.square().mean(0).max())
        MEASURED[f"{cell}: variance"] = (err, TOL)
        assert err <= TOL, f"{cell}: variance {err:.3e}"
        assert torch.equal(u.aleatoric_variance, torch.full_like(u.mean, 1.5 ** 2))
    calls = _calls(WF.LAUNCH_COUNTS)
    want = sums_calls(route, D, S)
    assert {k: calls.get(k, 0) for k in want} == want, (route, calls)
