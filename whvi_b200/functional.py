"""Autograd functions over the C ABI (libwhvi_b200.so): the fused WHVILinear layer, the
reparameterisation and the KL term.  PyTorch only owns the tensors, the autograd graph and
the stream; every FLOP of the hot path happens in the hand-written sm_100a kernels.

Shapes: ``x`` is ``(B, D)`` (one block shared by all MC samples -- the first WHVI layer of
a network) or ``(S, B, D)``; ``g`` is ``(S, D)``, one reparameterised vector per sample;
``s1, s2, bias`` are ``(D,)``; the output is ``(S, B, D)``.
"""
from __future__ import annotations

import ctypes
import functools

import torch
import torch.nn.functional as F
from torch.autograd import Function

from . import _lib

_WORKSPACES: dict[tuple[int, int], torch.Tensor] = {}

# Kernel-launch accounting (bench.py reads it): launches issued by each C-ABI call.
LAUNCH_COUNTS: dict[str, int] = {}
_LAUNCHES_PER_CALL = {"whvi_fwht_f32": 1, "whvi_fwht_f64": 1, "whvi_layer_fwd_f32": 1, "whvi_layer_bwd_f32": 3,
                      "whvi_layer_fwd_fused_f32": 1, "whvi_layer_bwd_fused_f32": 3,
                      "whvi_layer_bwd_scaled_f32": 3, "whvi_layer_loss_f32": 3, "whvi_reparam_f32": 1,
                      "whvi_reparam_bwd_f32": 1, "whvi_kl_f32": 1, "whvi_mc_moments_f32": 1,
                      "whvi_mc_moments_strided_f32": 1, "whvi_adam_f32": 1, "whvi_layer_moments_f32": 1,
                      "whvi_reparam_dense_f32": 2, "whvi_reparam_dense_bwd_f32": 1, "whvi_kl_dense_f32": 2,
                      "whvi_fwht_bf16": 1, "whvi_fwht_scaled_f32": 1, "whvi_layer_moments_add_f32": 1, "whvi_layer_fwd_bf16": 1, "whvi_column_fwd_f32": 3, "whvi_column_bwd_f32": 7, "whvi_pad_rows_f32": 1, "whvi_stacked_fwd_f32": 3, "whvi_stacked_bwd_f32": 6, "whvi_kl_grouped_f32": 1,
                      "whvi_layer_bwd_bf16": 3, "whvi_layer_loss_bf16": 3,
                      # dense grouped calls: the counts at D <= 64; at D >= 128 they run the tcgen05 sequence once per block
                      "whvi_reparam_dense_grouped_f32": 1, "whvi_reparam_dense_grouped_bwd_f32": 1, "whvi_kl_dense_grouped_f32": 2,
                      "whvi_stacked_fwd_g_f32": 2, "whvi_stacked_bwd_g_f32": 5, "whvi_column_fwd_g_f32": 2, "whvi_column_bwd_g_f32": 6,
                      # bf16 twins of the Stacked and Column calls: the fp32 calls' launches
                      "whvi_pad_rows_bf16": 1, "whvi_stacked_fwd_bf16": 3, "whvi_stacked_fwd_g_bf16": 2, "whvi_stacked_bwd_bf16": 6,
                      "whvi_stacked_bwd_g_bf16": 5, "whvi_column_fwd_bf16": 3, "whvi_column_fwd_g_bf16": 2, "whvi_column_bwd_bf16": 7,
                      "whvi_column_bwd_g_bf16": 6,
                      # categorical likelihood: the forward is the row kernel + the fixed-order sum of its per-CTA partials
                      "whvi_categorical_nll_f32": 2, "whvi_categorical_nll_bf16": 2, "whvi_categorical_nll_bwd_f32": 1,
                      "whvi_categorical_nll_bwd_bf16": 1, "whvi_categorical_predictive_f32": 1, "whvi_categorical_predictive_bf16": 1,
                      "whvi_im2col_f32": 1, "whvi_im2col_bf16": 1, "whvi_col2im_f32": 1, "whvi_col2im_bf16": 1}
# When set to a dict {"name": [(start_event, stop_event), ...]}, the named calls are bracketed
# by CUDA events on the launching stream (bench.py's per-kernel roofline timing).
EVENT_SINK: dict[str, list] | None = None


def _count(name: str) -> None:
    LAUNCH_COUNTS[name] = LAUNCH_COUNTS.get(name, 0) + _LAUNCHES_PER_CALL[name]


class _Timed:
    def __init__(self, name: str, tag: str = ""):
        self.name = name
        self.tag = tag   # position of the call in the model (bench.py's per-position roofline): "shared_x", "distinct_x/nodx" ...
        self.on = EVENT_SINK is not None and name in EVENT_SINK

    def __enter__(self):
        _count(self.name)
        if self.on:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if self.on:
            self.b.record()
            EVENT_SINK[self.name].append((self.a, self.b, self.tag))


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)   # the current stream's handle without a Stream object


def _stream(device: torch.device) -> int:
    if _raw_stream is not None:
        return _raw_stream(device.index if device.index is not None else torch.cuda.current_device())
    return torch.cuda.current_stream(device).cuda_stream


_capturing = getattr(torch._C, "_cuda_isCurrentStreamCapturing", None) or torch.cuda.is_current_stream_capturing


def _workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Per (device, stream) scratch buffer owned by PyTorch's caching allocator; the
    library itself never allocates.

    While a CUDA graph is being captured the buffer is a fresh tensor from the graph's own memory pool instead: a cached
    buffer would tie the graph to memory it does not own -- a buffer created during an EARLIER capture lives in that
    graph's pool (unmapped by the next ``empty_cache`` once that graph is gone, and ``torch.cuda.graph`` calls
    ``empty_cache`` on entry), and growing the cached buffer in the middle of a capture frees the one the kernels captured
    so far still point to.  Inside a capture the allocator reuses a freed scratch tensor for later allocations of the
    same graph in stream order, which is exactly the lifetime a workspace has."""
    if _capturing():
        return torch.empty(max(nbytes, 16), dtype=torch.uint8, device=device)
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream(device))
    buf = _WORKSPACES.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _WORKSPACES[key] = buf
    return buf


@functools.lru_cache(maxsize=None)
def _query(name: str, *dims) -> tuple:
    """Size queries of the C ABI (workspace bytes, partial-sum counts) are pure functions of the shape: asked once per shape,
    not once per call (a ctypes call with byref out-parameters costs ~4 us of host time)."""
    fn = getattr(_lib.lib(), name)
    if name == "whvi_layer_loss_sizes":
        a, b = ctypes.c_size_t(0), ctypes.c_int64(0)
        _lib.check(fn(*dims, ctypes.byref(a), ctypes.byref(b)), name)
        return a.value, b.value
    out = ctypes.c_int64(0) if name == "whvi_layer_fwd_partials" else ctypes.c_size_t(0)
    _lib.check(fn(*dims, ctypes.byref(out)), name)
    return (out.value,)


def _f32c(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.device.type != "cuda":
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name} must be float32 (got {t.dtype})")
    return t.contiguous()


def _bf16c(t: torch.Tensor, name: str) -> torch.Tensor:
    if t.device.type != "cuda":
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if t.dtype != torch.bfloat16:
        raise RuntimeError(f"{name} must be bfloat16 (got {t.dtype})")
    return t.contiguous()


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _layer_dims(x, g, s1, s2):
    if g.dim() != 2:
        raise RuntimeError("g must be (S, D)")
    S, D = g.shape
    if x.dim() == 2:
        B, xs = x.size(0), 0
    elif x.dim() == 3 and x.size(0) == S:
        B, xs = x.size(1), x.size(1) * D
    else:
        raise RuntimeError(f"x must be (B, D) or (S, B, D) with S = {S}; got {tuple(x.shape)}")
    if x.size(-1) != D or s1.numel() != D or s2.numel() != D:
        raise RuntimeError("last dimension of x, s1, s2 must equal D")
    return S, B, D, xs


def layer_forward_raw(x, g, s1, s2, bias=None, out=None, relu_out=False, target=None, from_t2=False):
    """y = s1 * H(g[s] * H(s2 * x)) (+bias) [-> max(y, 0)], no autograd.
    With ``target`` (B, D): returns ``(y, sum (y - target)^2)``, the sum as a 0-d tensor.
    ``from_t2``: ``x`` already holds ``H(s2 * x)`` (sample-independent), only the second half runs."""
    x, g, s1, s2 = _f32c(x, "x"), _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
    S, B, D, xs = _layer_dims(x, g, s1, s2)
    if bias is not None:
        bias = _f32c(bias, "bias").reshape(-1)
        if bias.numel() != D:
            raise RuntimeError("bias must have D elements")
    if out is None:
        out = torch.empty((S, B, D), dtype=torch.float32, device=x.device)
    L = _lib.lib()
    partials = None
    if target is not None:
        target = _f32c(target, "target")
        if target.shape != (B, D):
            raise RuntimeError(f"target must be {(B, D)}, got {tuple(target.shape)}")
        partials = torch.empty(max(_query("whvi_layer_fwd_partials", S, B, D)[0], 1), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device), _Timed("whvi_layer_fwd_fused_f32", ("shared_x" if xs == 0 else "distinct_x") + ("/from_t2" if from_t2 else "")):
        rc = L.whvi_layer_fwd_fused_f32(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(bias),
                                        out.data_ptr(), S, B, D, (1 if relu_out else 0) | (2 if from_t2 else 0),
                                        _ptr(target), _ptr(partials),
                                        _stream(x.device))
    _lib.check(rc, "whvi_layer_fwd_fused_f32")
    if target is not None:
        return out, partials.sum() if S * B > 0 else partials.sum() * 0
    return out


def layer_forward_bf16(x, g, s1, s2, bias=None, out=None, relu_out=False, from_t2=False):
    """The fused forward with bf16 activations in HBM (``whvi_layer_fwd_bf16``, SURVEY 8f N4): ``x`` (B, D) or (S, B, D) and
    the result are ``torch.bfloat16``; g, s1, s2, bias stay fp32 and so does every FLOP; the output is rounded once, at the
    store.  Inference only (no autograd): 4 B/element of activation traffic instead of 8."""
    if x.dtype != torch.bfloat16 or x.device.type != "cuda":
        raise RuntimeError("x must be a CUDA bfloat16 tensor")
    x = x.contiguous()
    g, s1, s2 = _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
    S, B, D, xs = _layer_dims(x, g, s1, s2)
    if bias is not None:
        bias = _f32c(bias, "bias").reshape(-1)
        if bias.numel() != D:
            raise RuntimeError("bias must have D elements")
    if out is None:
        out = torch.empty((S, B, D), dtype=torch.bfloat16, device=x.device)
    elif out.dtype != torch.bfloat16 or out.shape != (S, B, D) or not out.is_contiguous():
        raise RuntimeError("out must be a contiguous bfloat16 (S, B, D) tensor")
    with torch.cuda.device(x.device), _Timed("whvi_layer_fwd_bf16"):
        rc = _lib.lib().whvi_layer_fwd_bf16(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(bias), out.data_ptr(),
                                            S, B, D, (1 if relu_out else 0) | (2 if from_t2 else 0), _stream(x.device))
    _lib.check(rc, "whvi_layer_fwd_bf16")
    return out


def fwht_scaled_(x, scale, out=None):
    """out = H(scale * x) for a (D,) vector ``scale`` broadcast over the rows of ``x`` (rows, D), one pass
    (``whvi_fwht_scaled_f32``): the hoisted first transform t2 = H(s2 * x) of the MC predictive evaluation."""
    x, scale = _f32c(x, "x"), _f32c(scale, "scale").reshape(-1)
    if x.dim() != 2 or scale.numel() != x.size(1):
        raise RuntimeError("x must be (rows, D) and scale (D,)")
    if out is None:
        out = torch.empty_like(x)
    elif out.shape != x.shape or out.dtype != torch.float32 or not out.is_contiguous() or out.device != x.device:
        raise RuntimeError("out must be a contiguous float32 tensor of x's shape on the same device")
    with torch.cuda.device(x.device), _Timed("whvi_fwht_scaled_f32"):
        rc = _lib.lib().whvi_fwht_scaled_f32(x.data_ptr(), scale.data_ptr(), out.data_ptr(), x.size(0), x.size(1), _stream(x.device))
    _lib.check(rc, "whvi_fwht_scaled_f32")
    return out


def mc_moments_(y, sum_y, sum_y2=None, accumulate=True):
    """sum_y (+)= y.sum(0), sum_y2 (+)= (y*y).sum(0) over the leading MC-sample axis, in one pass
    over ``y`` (S, ...); samples ascending, bit-reproducible (SURVEY 8f N1)."""
    y = _f32c(y, "y")
    S = y.size(0)
    n = y[0].numel() if S > 0 else sum_y.numel()
    for t, name in ((sum_y, "sum_y"), (sum_y2, "sum_y2")):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n or t.device != y.device):
            raise RuntimeError(f"{name} must be a contiguous float32 tensor with {n} elements on {y.device}")
    with torch.cuda.device(y.device), _Timed("whvi_mc_moments_f32"):
        rc = _lib.lib().whvi_mc_moments_f32(y.data_ptr(), sum_y.data_ptr(), _ptr(sum_y2), S, n, 1 if accumulate else 0,
                                            _stream(y.device))
    _lib.check(rc, "whvi_mc_moments_f32")
    return sum_y, sum_y2


FUSED_MOMENTS_MIN_D, FUSED_MOMENTS_MAX_D = 8192, 32768


def layer_moments_raw(x, g, s1, s2, bias, sum_y, sum_y2=None, from_t2=False, accumulate=False, reserve_sms=0, init=None):
    """sum_y (+)= sum_s y[s], sum_y2 (+)= sum_s y[s]^2 for y[s] = s1 * H(g[s] * H(s2 * x)) + bias over ALL samples of ``g``
    in ONE kernel that keeps the running sums in tensor memory: no prediction is ever written to HBM
    (``whvi_layer_moments_f32``; 8192 <= D <= 32768).  ``x``: (B, D) shared or (S, B, D); ``from_t2``: x holds H(s2 * x);
    ``reserve_sms``: SMs the persistent grid leaves free for a collective kernel running next to it."""
    x, g, s1, s2 = _f32c(x, "x"), _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
    S, B, D, xs = _layer_dims(x, g, s1, s2)
    if bias is not None:
        bias = _f32c(bias, "bias").reshape(-1)
    for t, name in ((sum_y, "sum_y"), (sum_y2, "sum_y2")):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != B * D or t.device != x.device):
            raise RuntimeError(f"{name} must be a contiguous float32 tensor with {B * D} elements on {x.device}")
    flags = (2 if from_t2 else 0) | (4 if accumulate else 0) | ((int(reserve_sms) & 0xFF) << 8)
    if init is not None:   # (in_sum_y, in_sum_y2): out = in + this call's sums (``whvi_layer_moments_add_f32``)
        iy, iy2 = init
        with torch.cuda.device(x.device), _Timed("whvi_layer_moments_add_f32"):
            rc = _lib.lib().whvi_layer_moments_add_f32(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(bias),
                                                       _ptr(iy), _ptr(iy2), sum_y.data_ptr(), _ptr(sum_y2), S, B, D, flags, _stream(x.device))
        _lib.check(rc, "whvi_layer_moments_add_f32")
        return sum_y, sum_y2
    with torch.cuda.device(x.device), _Timed("whvi_layer_moments_f32", "from_t2" if from_t2 else "full"):
        rc = _lib.lib().whvi_layer_moments_f32(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(bias),
                                               sum_y.data_ptr(), _ptr(sum_y2), S, B, D, flags, _stream(x.device))
    _lib.check(rc, "whvi_layer_moments_f32")
    return sum_y, sum_y2


def mc_moments_into(y, in_y, in_y2, out_y, out_y2):
    """out = in + sum over the leading sample axis of ``y`` (and y^2).  ``y`` is (S, rows, D), possibly a
    block of rows of a larger contiguous (S, B, D) tensor; ``in_*`` may be None; ``out_*`` may be
    tensors that live on a peer GPU (symmetric memory): the scatter over NVLink is then part of
    the reduction kernel."""
    if y.dtype != torch.float32 or y.dim() != 3 or y.stride(2) != 1 or y.stride(1) != y.size(2):
        raise RuntimeError("y must be a float32 (S, rows, D) block with contiguous rows")
    S, n = y.size(0), y.size(1) * y.size(2)
    stride = y.stride(0) if S > 1 else n
    for t, name in ((in_y, "in_y"), (in_y2, "in_y2"), (out_y, "out_y"), (out_y2, "out_y2")):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n):
            raise RuntimeError(f"{name} must be a contiguous float32 tensor with {n} elements")
    with torch.cuda.device(y.device), _Timed("whvi_mc_moments_strided_f32"):
        rc = _lib.lib().whvi_mc_moments_strided_f32(y.data_ptr(), stride, _ptr(in_y), _ptr(in_y2), out_y.data_ptr(),
                                                    _ptr(out_y2), S, n, _stream(y.device))
    _lib.check(rc, "whvi_mc_moments_strided_f32")


@torch.no_grad()
def predictive_moments(x, mu, rho, s1, s2, bias=None, n_samples=64, chunk_samples=16, eps=None, generator=None,
                       sample_range=None, out=None, t2=None, scatter_to=None, L=None):
    """MC predictive mean and variance of one square WHVI layer (PAPER semantics) for inputs
    ``x`` (B, D) -- BASELINE config 5, what ``WHVIRegression.eval_model`` reduces
    ``WHVINetwork.forward``'s (B, out, S) output to (src/networks.py:36-54, :131-132) --
    without ever holding more than ``chunk_samples`` outputs:

    * t2 = H(s2 * x) once per input row (the first transform does not depend on the sample);
    * per sample chunk: g = mu + softplus(rho) * eps, y = s1 * H(g * t2) + bias (one transform
      per (sample, row)), then one pass that accumulates sum y and sum y^2.

    Returns ``(sum_y, sum_y2, S_done)`` as raw sums so that ranks holding different sample
    shards can all-reduce them (``distributed.reduce_predictive_moments``); ``sample_range``
    = (lo, hi) restricts this call to samples lo..hi-1 of ``eps`` / of the n_samples draws.
    ``out`` = (sum_y, sum_y2) buffers to overwrite (e.g. two halves of one all-reduce bucket).
    ``t2``: the hoisted transform ``fwht_(x * s2)`` if the caller already has it (``x`` may then be
    None) -- e.g. computed on row slices by different ranks and all-gathered.
    ``scatter_to``: [(row_lo, row_hi, out_y, out_y2), ...] covering all rows -- the LAST sample
    chunk's reduction writes its totals there instead of into the local sums (peer-GPU buffers of
    the ranks that own those rows; the experiment in ``tools/peer_moments.py`` uses it).
    ``L``: the dense posterior's lower-triangular factor (D, D) in place of ``rho``: g = mu + L eps per chunk
    (``reparam_dense``); the moments kernels are the same.
    """
    draw = (lambda e: ReparamFunction.apply(mu, rho, e)) if L is None else (lambda e: reparam_dense(mu, L, e))
    from .fwht import fwht_
    x = _f32c(x if t2 is None else t2, "x")
    if x.dim() != 2:
        raise RuntimeError("x must be (B, D)")
    B, D = x.shape
    lo, hi = sample_range if sample_range is not None else (0, n_samples if eps is None else eps.size(0))
    t2 = (fwht_scaled_(x, s2) if D >= 4 else fwht_(x * s2.reshape(1, D))) if t2 is None else x
    if out is not None:
        sum_y, sum_y2 = out
    else:
        sum_y = torch.empty((B, D), dtype=torch.float32, device=x.device)
        sum_y2 = torch.empty((B, D), dtype=torch.float32, device=x.device)
    if hi <= lo:
        sum_y.zero_(), sum_y2.zero_()
    if FUSED_MOMENTS_MIN_D <= D <= FUSED_MOMENTS_MAX_D and scatter_to is None and hi > lo:
        # one kernel for all samples: running sums in tensor memory, nothing but the two results goes to HBM
        e = eps[lo:hi] if eps is not None else torch.randn((hi - lo, D), device=x.device, generator=generator)
        g = draw(e.contiguous())
        layer_moments_raw(t2, g, s1, s2, bias, sum_y, sum_y2, from_t2=True, accumulate=False)
        return sum_y, sum_y2, hi - lo
    ybuf = torch.empty((min(chunk_samples, max(hi - lo, 1)), B, D), dtype=torch.float32, device=x.device)
    for s0 in range(lo, hi, chunk_samples):
        s1_ = min(s0 + chunk_samples, hi)
        e = eps[s0:s1_] if eps is not None else torch.randn((s1_ - s0, D), device=x.device, generator=generator)
        g = draw(e.contiguous())
        y = layer_forward_raw(t2, g, s1, s2, bias, out=ybuf[: s1_ - s0], from_t2=True)
        if scatter_to is not None and s1_ == hi:
            for r0, r1, oy, oy2 in scatter_to:
                mc_moments_into(y[:, r0:r1], sum_y[r0:r1] if s0 > lo else None, sum_y2[r0:r1] if s0 > lo else None, oy, oy2)
        else:
            mc_moments_(y, sum_y, sum_y2, accumulate=s0 > lo)   # the first chunk overwrites: no zero-fill pass
    return sum_y, sum_y2, hi - lo


FUSED_BWD_MAX_D = 8192   # a row pair, its transposition buffers and two pipeline stages fill an SM's shared memory there


@torch.no_grad()
def _layer_backward_multipass(x, dy, g, s1, s2, want_dx, want_dbias, relu_in, target, coef, dy_scale):
    """D = 2^14, 2^15 (the config-5 width): the backward as four passes of the batched FWHT kernel (``whvi_fwht_f32``) per
    MC sample with the elementwise products and column sums between them as tensor ops -- the same math as the fused
    kernel (SURVEY App. A), ~6x its HBM traffic, O(B.D) extra memory.  The reference's autograd has no width limit
    (``src/fwht/cuda/fwht.py:14-16``), so neither has the drop-in; the fused single-pass kernels stop at 8192."""
    from .fwht import fwht_
    S, D = g.shape
    shared = x.dim() == 2
    B = x.size(0) if shared else x.size(1)
    dev = x.device
    dx = torch.empty((S, B, D), dtype=torch.float32, device=dev) if want_dx else None
    dg = torch.empty((S, D), dtype=torch.float32, device=dev)
    ds1, ds2 = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    dbias = torch.zeros(D, device=dev) if want_dbias else None
    buf = torch.empty((B, D), dtype=torch.float32, device=dev)
    for s in range(S):
        xs_ = x if shared else x[s]
        if target is not None:
            dys = coef * (dy[s] - target)
        elif dy_scale is not None:
            dys = dy_scale.reshape(()) * dy[s]
        else:
            dys = dy[s]
        t2 = fwht_(xs_ * s2)
        dt3 = fwht_(dys * s1, out=buf)
        dg[s] = (dt3 * t2).sum(dim=0)
        dt1 = fwht_(dt3 * g[s], out=buf)
        ds2 += (dt1 * xs_).sum(dim=0)
        if want_dx:
            torch.mul(dt1, s2, out=dx[s])
            if relu_in:
                dx[s].mul_(xs_ > 0)
        t4 = fwht_(t2.mul_(g[s]), out=buf)
        ds1 += (dys * t4).sum(dim=0)
        if want_dbias:
            dbias += dys.sum(dim=0)
    return dx, dg, ds1, ds2, dbias


def layer_backward_raw(x, dy, g, s1, s2, want_dx=True, want_dbias=False, relu_in=False, target=None, coef=None,
                       dy_scale=None):
    """Returns (dx | None, dg, ds1, ds2, dbias | None); dx is (S,B,D) even for shared x.
    ``relu_in``: x came out of a fused ReLU, dx is masked by x > 0.  ``target``/``coef``:
    ``dy`` holds the layer's saved output and the upstream gradient is
    coef * (output - target) formed inside the kernel (coef: 0-d / 1-element CUDA tensor).
    A bfloat16 ``x`` selects the bf16-activation backward (``layer_backward_bf16``)."""
    if x.dtype == torch.bfloat16:
        if target is not None:
            raise RuntimeError("the backward from the saved output and a target (RESID) is fp32 only; bf16 activations "
                               "take the unfused route")
        return layer_backward_bf16(x, dy, g, s1, s2, want_dx, want_dbias, relu_in, dy_scale)
    x, dy, g, s1, s2 = _f32c(x, "x"), _f32c(dy, "dy"), _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
    S, B, D, xs = _layer_dims(x, g, s1, s2)
    if dy.shape != (S, B, D):
        raise RuntimeError(f"dy must be {(S, B, D)}, got {tuple(dy.shape)}")
    dev = x.device
    if target is not None:
        target, coef = _f32c(target, "target"), _f32c(coef, "coef").reshape(1)
    if D > FUSED_BWD_MAX_D:
        return _layer_backward_multipass(x, dy, g, s1, s2, want_dx, want_dbias, relu_in, target, coef, dy_scale)
    dx = torch.empty((S, B, D), dtype=torch.float32, device=dev) if want_dx else None
    dg = torch.empty((S, D), dtype=torch.float32, device=dev)
    ds1 = torch.empty(D, dtype=torch.float32, device=dev)
    ds2 = torch.empty(D, dtype=torch.float32, device=dev)
    dbias = torch.empty(D, dtype=torch.float32, device=dev) if want_dbias else None
    L = _lib.lib()
    ws = _workspace(dev, _query("whvi_layer_bwd_workspace_bytes", S, B, D)[0])
    if dy_scale is not None:  # upstream gradient = dy_scale * dy (see WHVILayerLossFunction)
        if target is not None:
            raise RuntimeError("dy_scale and target are mutually exclusive")
        dy_scale = _f32c(dy_scale, "dy_scale").reshape(1)
        with torch.cuda.device(dev), _Timed("whvi_layer_bwd_scaled_f32", ("shared_x" if xs == 0 else "distinct_x") + ("" if want_dx else "/nodx")):
            rc = L.whvi_layer_bwd_scaled_f32(x.data_ptr(), xs, dy.data_ptr(), dy_scale.data_ptr(), g.data_ptr(),
                                             s1.data_ptr(), s2.data_ptr(), _ptr(dx), dg.data_ptr(), ds1.data_ptr(),
                                             ds2.data_ptr(), _ptr(dbias), ws.data_ptr(), ws.numel(), S, B, D,
                                             1 if relu_in else 0, _stream(dev))
        _lib.check(rc, "whvi_layer_bwd_scaled_f32")
        return dx, dg, ds1, ds2, dbias
    with torch.cuda.device(dev), _Timed("whvi_layer_bwd_fused_f32", ("shared_x" if xs == 0 else "distinct_x") + ("" if want_dx else "/nodx")):
        rc = L.whvi_layer_bwd_fused_f32(x.data_ptr(), xs, dy.data_ptr(), g.data_ptr(), s1.data_ptr(), s2.data_ptr(),
                                        _ptr(dx), dg.data_ptr(), ds1.data_ptr(), ds2.data_ptr(), _ptr(dbias),
                                        ws.data_ptr(), ws.numel(), S, B, D, 1 if relu_in else 0, _ptr(target),
                                        _ptr(coef), _stream(dev))
    _lib.check(rc, "whvi_layer_bwd_fused_f32")
    return dx, dg, ds1, ds2, dbias


def layer_backward_bf16(x, dy, g, s1, s2, want_dx=True, want_dbias=False, relu_in=False, dy_scale=None):
    """``layer_backward_raw`` with bf16 activations (``whvi_layer_bwd_bf16``): ``x``, ``dy`` and the returned dx are
    ``torch.bfloat16``; g, s1, s2, dy_scale and dg, ds1, ds2, dbias are fp32.  Defined as the fp32 backward on the widened
    inputs: dx = bf16(dx_f32), rounded once; the parameter gradients are bit-identical to the fp32 call's."""
    x, dy = _bf16c(x, "x"), _bf16c(dy, "dy")
    g, s1, s2 = _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
    S, B, D, xs = _layer_dims(x, g, s1, s2)
    if dy.shape != (S, B, D):
        raise RuntimeError(f"dy must be {(S, B, D)}, got {tuple(dy.shape)}")
    if dy_scale is not None:
        dy_scale = _f32c(dy_scale, "dy_scale").reshape(1)
    if D > FUSED_BWD_MAX_D:   # the fp32 multi-pass backward on the widened inputs, dx rounded once at the end
        dx, dg, ds1, ds2, dbias = _layer_backward_multipass(x.float(), dy.float(), g, s1, s2, want_dx, want_dbias, relu_in,
                                                            None, None, dy_scale)
        return (None if dx is None else dx.to(torch.bfloat16)), dg, ds1, ds2, dbias
    if (B * D) % 8 != 0:
        # D = 4 with an odd B: the kernel's bulk copies move whole 16-byte units per sample; one zero row of x and dy adds
        # zero to every parameter gradient, so the padded call is exact
        x, dy = F.pad(x, (0, 0, 0, 1)), F.pad(dy, (0, 0, 0, 1))
        dx, dg, ds1, ds2, dbias = layer_backward_bf16(x, dy, g, s1, s2, want_dx, want_dbias, relu_in, dy_scale)
        return (None if dx is None else dx[:, :B].contiguous()), dg, ds1, ds2, dbias
    dev = x.device
    dx = torch.empty((S, B, D), dtype=torch.bfloat16, device=dev) if want_dx else None
    dg = torch.empty((S, D), dtype=torch.float32, device=dev)
    ds1 = torch.empty(D, dtype=torch.float32, device=dev)
    ds2 = torch.empty(D, dtype=torch.float32, device=dev)
    dbias = torch.empty(D, dtype=torch.float32, device=dev) if want_dbias else None
    ws = _workspace(dev, _query("whvi_layer_bwd_workspace_bytes", S, B, D)[0])
    with torch.cuda.device(dev), _Timed("whvi_layer_bwd_bf16", ("shared_x" if xs == 0 else "distinct_x") + ("" if want_dx else "/nodx")):
        rc = _lib.lib().whvi_layer_bwd_bf16(x.data_ptr(), xs, dy.data_ptr(), _ptr(dy_scale), g.data_ptr(), s1.data_ptr(),
                                            s2.data_ptr(), _ptr(dx), dg.data_ptr(), ds1.data_ptr(), ds2.data_ptr(), _ptr(dbias),
                                            ws.data_ptr(), ws.numel(), S, B, D, 1 if relu_in else 0, _stream(dev))
    _lib.check(rc, "whvi_layer_bwd_bf16")
    return dx, dg, ds1, ds2, dbias


LOSS_LAYER_MIN_D, LOSS_LAYER_MAX_D = 128, 4096

class DeferredScale:
    """Scalar hand-over between two autograd nodes of ONE graph: the fused loss layer computes its
    dx for a unit loss coefficient and leaves the true coefficient here; the producer of its input
    (a fused ``WHVILayerFunction``) picks it up in its own backward and applies it while loading dy
    (``whvi_layer_bwd_scaled_f32``), which saves a pass over dx.  ``WHVINetwork._run`` creates one
    holder per (producer, loss layer) pair and passes it to both ``forward`` calls, so the scale is
    carried by the graph itself: copies of the gradient tensor (hooks, accumulation) cannot lose
    it, and nothing outlives the graph.  If the consumer's backward has not run when the producer's
    does (``torch.autograd.grad`` on a subset), the holder is empty and dy is used as it is."""

    __slots__ = ("value",)

    def __init__(self):
        self.value = None

    def put(self, c: torch.Tensor) -> None:
        self.value = c

    def take(self):
        c, self.value = self.value, None
        return c


def layer_loss_raw(x, g, s1, s2, bias, target, want_dx=True, relu_in=False):
    """Fused last layer (forward + squared-error residual + backward for a unit coefficient).
    Returns (sum r^2 as a 0-d tensor, dx | None, dg, ds1, ds2, dbias | None).
    A bfloat16 ``x`` selects ``whvi_layer_loss_bf16``: dx is then bf16 (rounded once), everything else as in fp32."""
    bf16 = x.dtype == torch.bfloat16
    x = _bf16c(x, "x") if bf16 else _f32c(x, "x")
    g, s1, s2 = _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
    S, B, D, xs = _layer_dims(x, g, s1, s2)
    target = _f32c(target, "target")
    if target.shape != (B, D):
        raise RuntimeError(f"target must be {(B, D)}, got {tuple(target.shape)}")
    if bias is not None:
        bias = _f32c(bias, "bias").reshape(-1)
    dev = x.device
    L = _lib.lib()
    need, nsq = _query("whvi_layer_loss_sizes", S, B, D)
    ws = _workspace(dev, need)
    sqp = torch.zeros(max(nsq, 1), dtype=torch.float32, device=dev)   # an upper bound: unused entries stay zero
    dx = torch.empty((S, B, D), dtype=x.dtype, device=dev) if want_dx else None
    dg = torch.empty((S, D), dtype=torch.float32, device=dev)
    ds1 = torch.empty(D, dtype=torch.float32, device=dev)
    ds2 = torch.empty(D, dtype=torch.float32, device=dev)
    dbias = torch.empty(D, dtype=torch.float32, device=dev) if bias is not None else None
    name = "whvi_layer_loss_bf16" if bf16 else "whvi_layer_loss_f32"
    with torch.cuda.device(dev), _Timed(name, ("shared_x" if xs == 0 else "distinct_x") + ("" if want_dx else "/nodx")):
        rc = getattr(L, name)(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(bias),
                              target.data_ptr(), _ptr(dx), dg.data_ptr(), ds1.data_ptr(), ds2.data_ptr(),
                              _ptr(dbias), sqp.data_ptr(), ws.data_ptr(), ws.numel(), S, B, D,
                              1 if relu_in else 0, _stream(dev))
    _lib.check(rc, name)
    return sqp.sum(), dx, dg, ds1, ds2, dbias


class WHVILayerFunction(Function):
    """y[s,b] = s1 * H(g[s] * H(s2 * x[s,b])) (+ bias) with the fused backward.

    ``relu_out``: the ReLU that follows the layer is applied inside the forward kernel.
    ``relu_in``: the input is the output of such a fused ReLU; the backward kernel masks
    dx by x > 0, i.e. returns the gradient w.r.t. the PRODUCER's pre-activation.  The two
    flags are set in matching pairs by ``WHVINetwork`` (producer relu_out <-> consumer
    relu_in), which is what makes the chain rule come out right without the ReLU ever
    touching HBM.

    A bfloat16 ``x`` runs the bf16-activation kernels (output and dx bf16, parameter gradients fp32); the shared-input
    transform is not hoisted then, because a bf16 t2 would add a rounding the fp32 composition does not have."""

    @staticmethod
    def forward(ctx, x, g, s1, s2, bias, relu_out=False, relu_in=False, dy_scale_from=None):
        if x.dtype == torch.bfloat16:
            y = layer_forward_bf16(x, g, s1, s2, bias, relu_out=relu_out)
        elif x.dim() == 2 and g.size(0) >= 4 and g.size(-1) >= 128 and g.size(0) * x.numel() >= HOIST_MIN_ELEMENTS:
            # one (B, D) input block for all samples (the first layer of a network): the first transform does not depend
            # on the sample (SURVEY 8d C5), so it is done once -- t2 = H(s2 * x), one pass over B * D elements -- and every
            # (sample, row) pair costs one transform; the output stream is the same, the kernel 12% shorter (D = 4096)
            y = layer_forward_raw(fwht_scaled_(x, s2), g, s1, s2, bias, relu_out=relu_out, from_t2=True)
        else:
            y = layer_forward_raw(x, g, s1, s2, bias, relu_out=relu_out)
        ctx.save_for_backward(x, g, s1, s2)
        ctx.has_bias = bias is not None
        ctx.relu_in = relu_in
        ctx.dy_scale_from = dy_scale_from  # DeferredScale shared with the fused loss layer that consumes y
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g, s1, s2 = ctx.saved_tensors
        want_dx = ctx.needs_input_grad[0]
        want_db = ctx.has_bias and ctx.needs_input_grad[4]
        # dy came from a fused loss layer that left its loss coefficient in the shared holder
        scale = ctx.dy_scale_from.take() if ctx.dy_scale_from is not None else None
        dx, dg, ds1, ds2, dbias = layer_backward_raw(x, dy.contiguous(), g, s1, s2, want_dx=want_dx, want_dbias=want_db,
                                                     relu_in=ctx.relu_in, dy_scale=scale)
        if dx is not None and x.dim() == 2:
            dx = dx.sum(dim=0)
        return dx, dg, ds1, ds2, dbias, None, None, None


MIN_LAYER_D = 4  # narrowest row the layer kernels take (one float4)
HOIST_MIN_ELEMENTS = 1 << 24   # S * B * D from which hoisting the shared-input transform pays for its extra launch (measured
                               # for D = 1024, 4096, 8192; not applied below D = 128)


def whvi_layer(x, g, s1, s2, bias=None, relu_out=False, relu_in=False, dy_scale_from=None):
    D = g.size(-1)
    if D < MIN_LAYER_D:
        # D = 1, 2 (the reference takes them, e.g. WHVILinear(2, 2) on 2-D toy inputs): zero-pad x, g, s1, s2 to
        # width 4.  H_4 = H_2 (x) H_2 and the padded s2 / g / s1 zero the other block at every stage, so the first D
        # outputs -- and, through autograd of the pad, all gradients -- are exactly the width-D layer's.
        pad = lambda v: None if v is None else torch.nn.functional.pad(v, (0, MIN_LAYER_D - D))
        y = WHVILayerFunction.apply(pad(x), pad(g), pad(s1), pad(s2), pad(bias), relu_out, relu_in, dy_scale_from)
        return y[..., :D]
    return WHVILayerFunction.apply(x, g, s1, s2, bias, relu_out, relu_in, dy_scale_from)


class WHVILayerSqErrFunction(Function):
    """Last layer of a regression net fused with the data term of the Gaussian MNLL:
    returns ``(y_hat, sum (y_hat - target)^2)``.  The squared-error sum is reduced inside the
    forward kernel, and in the backward the upstream gradient 2*d_sq*(y_hat - target) is
    formed inside the backward kernel from the saved output -- no dy tensor, no separate
    elementwise passes (reference: src/likelihoods.py:18-29 on top of src/weights.py:87-93)."""

    @staticmethod
    def forward(ctx, x, g, s1, s2, bias, target, relu_in=False):
        y, sq = layer_forward_raw(x, g, s1, s2, bias, target=target)
        ctx.save_for_backward(x, g, s1, s2, y, target)
        ctx.has_bias = bias is not None
        ctx.relu_in = relu_in
        ctx.set_materialize_grads(False)
        return y, sq

    @staticmethod
    def backward(ctx, d_y, d_sq):
        x, g, s1, s2, y, target = ctx.saved_tensors
        want_dx = ctx.needs_input_grad[0]
        want_db = ctx.has_bias and ctx.needs_input_grad[4]
        if d_sq is None:
            d_sq = torch.zeros((), device=x.device)
        if d_y is None:   # the usual case: the predictions feed nothing but the loss
            dx, dg, ds1, ds2, dbias = layer_backward_raw(x, y, g, s1, s2, want_dx=want_dx, want_dbias=want_db,
                                                         relu_in=ctx.relu_in, target=target,
                                                         coef=(2.0 * d_sq).to(torch.float32))
        else:
            dy = d_y + 2.0 * d_sq * (y - target)
            dx, dg, ds1, ds2, dbias = layer_backward_raw(x, dy, g, s1, s2, want_dx=want_dx, want_dbias=want_db,
                                                         relu_in=ctx.relu_in)
        if dx is not None and x.dim() == 2:
            dx = dx.sum(dim=0)
        return dx, dg, ds1, ds2, dbias, None, None


def whvi_layer_sqerr(x, g, s1, s2, bias, target, relu_in=False):
    return WHVILayerSqErrFunction.apply(x, g, s1, s2, bias, target, relu_in)


class WHVILayerLossFunction(Function):
    """Training-time last layer fused with the Gaussian-MNLL data term: returns only
    ``sum (y_hat - target)^2``; the predictions never exist in HBM and the layer's whole backward
    is computed in the same pass (for a unit loss coefficient) and kept for ``backward``.

    ``dx_scale_to``: a ``DeferredScale`` shared with the fused ``WHVILayerFunction`` that produced
    ``x`` and is its ONLY consumer (set by ``WHVINetwork._run`` in matching pairs, like
    relu_out/relu_in); ``dx`` is then handed on unscaled, the coefficient goes into the holder and
    the producer's backward kernel applies it on load, saving a pass over dx.

    bf16 ``x``: dx is bf16, rounded once by the kernel for the unit coefficient.  Handed on through ``dx_scale_to`` it is
    scaled in fp32 inside the producer's backward, so the chain rounds once per layer boundary.  Without a holder (shared
    x, a producer without the fused ReLU, a non-square producer) the coefficient is applied here to the bf16 dx, which
    rounds a second time: bf16(bf16(dx) * c)."""

    @staticmethod
    def forward(ctx, x, g, s1, s2, bias, target, relu_in=False, dx_scale_to=None):
        want_dx = ctx.needs_input_grad[0]
        sq, dx, dg, ds1, ds2, dbias = layer_loss_raw(x, g, s1, s2, bias, target, want_dx=want_dx, relu_in=relu_in)
        ctx.shared_x = x.dim() == 2
        ctx.dx_scale_to = dx_scale_to if (want_dx and not ctx.shared_x) else None
        ctx.has_dx, ctx.has_db = dx is not None, dbias is not None
        ctx.save_for_backward(*[t for t in (dx, dg, ds1, ds2, dbias) if t is not None])
        return sq

    @staticmethod
    def backward(ctx, d_sq):
        saved = list(ctx.saved_tensors)
        dx = saved.pop(0) if ctx.has_dx else None
        dg, ds1, ds2 = saved[0], saved[1], saved[2]
        dbias = saved[3] if ctx.has_db else None
        c = (2.0 * d_sq).to(torch.float32)
        if dx is not None:
            if ctx.shared_x:
                dx = dx.sum(dim=0) * c
            elif ctx.dx_scale_to is not None:
                ctx.dx_scale_to.put(c.reshape(1))
            else:
                dx = dx.mul_(c)
        return dx, dg * c, ds1 * c, ds2 * c, None if dbias is None else dbias * c, None, None, None


def whvi_layer_loss(x, g, s1, s2, bias, target, relu_in=False, dx_scale_to=None):
    return WHVILayerLossFunction.apply(x, g, s1, s2, bias, target, relu_in, dx_scale_to)


class ReparamFunction(Function):
    """g[s] = mu + softplus(rho) * eps[s]  (src/weights.py:43-50, :82-83)."""

    @staticmethod
    def forward(ctx, mu, rho, eps):
        mu, rho, eps = _f32c(mu, "g_mu"), _f32c(rho, "g_rho"), _f32c(eps, "eps")
        S, D = eps.shape
        g = torch.empty_like(eps)
        with torch.cuda.device(eps.device), _Timed("whvi_reparam_f32"):
            rc = _lib.lib().whvi_reparam_f32(mu.data_ptr(), rho.data_ptr(), eps.data_ptr(), g.data_ptr(), S, D, 0,
                                             _stream(eps.device))
        _lib.check(rc, "whvi_reparam_f32")
        ctx.save_for_backward(rho, eps)
        return g

    @staticmethod
    def backward(ctx, dg):
        rho, eps = ctx.saved_tensors
        dg = _f32c(dg, "dg")
        S, D = eps.shape
        dmu = torch.empty(D, dtype=torch.float32, device=eps.device)
        drho = torch.empty(D, dtype=torch.float32, device=eps.device)
        with torch.cuda.device(eps.device), _Timed("whvi_reparam_bwd_f32"):
            rc = _lib.lib().whvi_reparam_bwd_f32(rho.data_ptr(), eps.data_ptr(), dg.data_ptr(), dmu.data_ptr(),
                                                 drho.data_ptr(), S, D, 0, 0, _stream(eps.device))
        _lib.check(rc, "whvi_reparam_bwd_f32")
        return dmu, drho, None


def reparam(mu, rho, eps):
    return ReparamFunction.apply(mu, rho, eps)


def _blocks(tensors, name):
    """(base, stride): G blocks' parameters read where they lie when evenly spaced (FlatParams, a module's own packing),
    else a stacked copy."""
    base = _f32c(tensors[0], name)
    if len(tensors) == 1:
        return base.detach(), base.numel()
    stride = uniform_stride(tensors)
    if stride is None or any(t.dtype != torch.float32 for t in tensors):
        return torch.stack([_f32c(t, name).detach() for t in tensors]), base.numel()
    return base.detach(), stride


class ReparamDenseFunction(Function):
    """g[k, s] = mu_k + L_k eps[k, s] for G blocks with dense lower-triangular L_k (D, D), D <= 64 or a multiple of 128: superset of the
    reference (whose posterior is diagonal, SURVEY F5).  ``eps`` (G, S, D); ``params`` = G x mu, G x L (the blocks' own
    parameters).  One C call per direction (``whvi_reparam_dense_grouped_f32`` / ``..._bwd_f32``): the CUDA-core kernels at
    D <= 64, the tcgen05 GEMMs of ``csrc/reparam_dense.cu`` block after block at D >= 128 (g = mu + E L^T, dL = tril(dg^T E)),
    dmu a device column sum."""

    @staticmethod
    def forward(ctx, eps, *params):
        G = len(params) // 2
        eps = _f32c(eps, "eps")
        if eps.dim() != 3 or eps.size(0) != G:
            raise RuntimeError(f"eps must be ({G}, S, D), got {tuple(eps.shape)}")
        _, S, D = eps.shape
        if any(m.numel() != D for m in params[:G]) or any(tuple(l.shape) != (D, D) for l in params[G:]):
            raise RuntimeError(f"every g_mu must have {D} elements and every g_L be {(D, D)}")
        mu, mu_stride = _blocks(params[:G], "g_mu")
        L, L_stride = _blocks(params[G:], "g_L")
        g = torch.empty_like(eps)
        with torch.cuda.device(eps.device):
            ws = _workspace(eps.device, _query("whvi_reparam_dense_grouped_workspace_bytes", S, D)[0])
            with _Timed("whvi_reparam_dense_grouped_f32", f"D={D},G={G}"):
                rc = _lib.lib().whvi_reparam_dense_grouped_f32(mu.data_ptr(), mu_stride, L.data_ptr(), L_stride, eps.data_ptr(), g.data_ptr(),
                                                               S, D, G, ws.data_ptr(), ws.numel(), _stream(eps.device))
        _lib.check(rc, "whvi_reparam_dense_grouped_f32")
        ctx.save_for_backward(eps)
        return g

    @staticmethod
    def backward(ctx, dg):
        (eps,) = ctx.saved_tensors
        dg = _f32c(dg, "dg")
        G, S, D = eps.shape
        dmu = torch.empty((G, D), dtype=torch.float32, device=eps.device)
        dL = torch.empty((G, D, D), dtype=torch.float32, device=eps.device)
        with torch.cuda.device(eps.device):
            ws = _workspace(eps.device, _query("whvi_reparam_dense_grouped_workspace_bytes", S, D)[0])
            with _Timed("whvi_reparam_dense_grouped_bwd_f32", f"D={D},G={G}"):
                rc = _lib.lib().whvi_reparam_dense_grouped_bwd_f32(eps.data_ptr(), dg.data_ptr(), dmu.data_ptr(), dL.data_ptr(), S, D, G,
                                                                   ws.data_ptr(), ws.numel(), _stream(eps.device))
        _lib.check(rc, "whvi_reparam_dense_grouped_bwd_f32")
        return (None, *dmu.unbind(0), *dL.unbind(0))


def reparam_dense_grouped(mus, Ls, eps):
    """(G, S, D) samples of G dense blocks for noise ``eps`` (G, S, D)."""
    return ReparamDenseFunction.apply(eps, *mus, *Ls)


def reparam_dense(mu, L, eps):
    """g[s] = mu + L eps[s] for one block: eps, g (S, D)."""
    return ReparamDenseFunction.apply(eps.unsqueeze(0), mu, L)[0]


class KLDenseFunction(Function):
    """KL( N(mu, L L^T) || N(0, lambda I) ) = 0.5 (D ln lambda - 2 sum ln L_ii - D + |L|_F^2 / lambda + |mu|^2 / lambda) with its
    gradients in one pass over L (north-star kernel (5), dense form: the log-determinant is 2 sum ln L_ii)."""

    @staticmethod
    def forward(ctx, mu, L, lambda_):
        mu, L = _f32c(mu, "g_mu"), _f32c(L, "g_L")
        D = mu.numel()
        if L.shape != (D, D):
            raise RuntimeError(f"L must be {(D, D)}, got {tuple(L.shape)}")
        out = torch.empty(1, dtype=torch.float32, device=mu.device)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        dmu = torch.empty_like(mu) if need_grad else None
        dL = torch.empty_like(L) if need_grad else None
        ws = torch.empty(D, dtype=torch.float64, device=mu.device)
        with torch.cuda.device(mu.device), _Timed("whvi_kl_dense_f32"):
            rc = _lib.lib().whvi_kl_dense_f32(mu.data_ptr(), L.data_ptr(), float(lambda_), D, out.data_ptr(), _ptr(dmu), _ptr(dL),
                                              1.0, ws.data_ptr(), ws.numel() * 8, _stream(mu.device))
        _lib.check(rc, "whvi_kl_dense_f32")
        if need_grad:
            ctx.save_for_backward(dmu, dL)
        return out.reshape(())

    @staticmethod
    def backward(ctx, dkl):
        dmu, dL = ctx.saved_tensors
        return dmu * dkl, dL * dkl, None


def kl_gaussian_dense(mu, L, lambda_):
    return KLDenseFunction.apply(mu, L, lambda_)


class KLDenseGroupedFunction(Function):
    """Sum over G blocks of the dense KL term with all gradients, one C call (``whvi_kl_dense_grouped_f32``)."""

    @staticmethod
    def forward(ctx, lambda_, *params):
        G = len(params) // 2
        mu, mu_stride = _blocks(params[:G], "g_mu")
        L, L_stride = _blocks(params[G:], "g_L")
        D = params[0].numel()
        dev = mu.device
        out = torch.empty(1, dtype=torch.float32, device=dev)
        need_grad = any(ctx.needs_input_grad[1:])
        dmu = torch.empty((G, D), dtype=torch.float32, device=dev) if need_grad else None
        dL = torch.empty((G, D, D), dtype=torch.float32, device=dev) if need_grad else None
        ws = torch.empty(G * D, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev), _Timed("whvi_kl_dense_grouped_f32", f"D={D},G={G}"):
            rc = _lib.lib().whvi_kl_dense_grouped_f32(mu.data_ptr(), mu_stride, L.data_ptr(), L_stride, float(lambda_), D, G, out.data_ptr(),
                                                      _ptr(dmu), _ptr(dL), 1.0, ws.data_ptr(), ws.numel() * 8, _stream(dev))
        _lib.check(rc, "whvi_kl_dense_grouped_f32")
        ctx.G = G
        if need_grad:
            ctx.save_for_backward(dmu, dL)
        return out.reshape(())

    @staticmethod
    def backward(ctx, dkl):
        dmu, dL = ctx.saved_tensors
        return (None, *(dmu * dkl).unbind(0), *(dL * dkl).unbind(0))


def kl_gaussian_dense_grouped(mus, Ls, lambda_):
    return KLDenseGroupedFunction.apply(lambda_, *mus, *Ls)


# ---------------------------------------------------------------------------------------------- Stacked layer, one call per direction
def uniform_stride(tensors) -> int | None:
    """Floats between consecutive tensors' first elements when they are evenly spaced in memory (stride >= numel, a multiple
    of 4), else None.  The blocks' separate nn.Parameters are evenly spaced once packed (FlatParams, or the Stacked module's
    own packing), and then the kernels read them where they lie."""
    if len(tensors) == 1:
        return tensors[0].numel()
    p0 = tensors[0].data_ptr()
    step = tensors[1].data_ptr() - p0
    if step < 4 * tensors[0].numel() or step % 16 != 0:
        return None
    for k, t in enumerate(tensors):
        if t.data_ptr() != p0 + k * step or not t.is_contiguous():
            return None
    return step // 4


def _act(t: torch.Tensor, name: str) -> torch.Tensor:
    """A contiguous fp32 or bf16 CUDA activation (the Stacked and Column calls take either, dispatching on the dtype)."""
    return _bf16c(t, name) if t.dtype == torch.bfloat16 else _f32c(t, name)


def _stacked_input(x, S, D):
    """(x zero-padded to D columns, B, x_sample_stride) for a Stacked call (src/weights.py:197-198); fp32 or bf16, as x."""
    n_in = x.size(-1)
    if n_in < D:
        name = "whvi_pad_rows_bf16" if x.dtype == torch.bfloat16 else "whvi_pad_rows_f32"
        xp = torch.empty(x.shape[:-1] + (D,), dtype=x.dtype, device=x.device)
        with _Timed(name):
            _lib.check(getattr(_lib.lib(), name)(x.data_ptr(), xp.data_ptr(), x.numel() // n_in, n_in, D, _stream(x.device)), name)
    else:
        xp = x
    if xp.dim() == 2:
        return xp, xp.size(0), 0
    if xp.dim() == 3 and xp.size(0) == S:
        return xp, xp.size(1), xp.size(1) * D
    raise RuntimeError(f"x must be (B, n_in) or (S, B, n_in) with S = {S}; got {tuple(x.shape)}")


def _stacked_vectors(groups, D):
    """The blocks' (D,) parameter vectors, one list of G tensors per kind, as one base tensor per kind and ONE stride shared
    by all kinds: read where they lie when they are evenly spaced alike, else a (kinds, G, D) copy."""
    strides = [uniform_stride(g_) for g_ in groups]
    if any(v is None for v in strides) or len(set(strides)) != 1:
        packed = torch.stack([torch.stack([t.detach().reshape(-1) for t in g_]) for g_ in groups])
        return list(packed.unbind(0)), D
    return [g_[0].detach() for g_ in groups], strides[0]


def _stacked_bwd_rows(xp, xs, dy, B, D):
    """bf16 at D = 4 with an odd B: the backward's bulk copies move whole 16-byte units per sample, so the call gets one zero row
    of the padded x and of dy (as ``layer_backward_bf16``), which adds zero to every gradient; the caller drops dx's extra row.
    Returns (xp, xs, dy, B) for the call."""
    if xp.dtype != torch.bfloat16 or (B * D) % 8 == 0:
        return xp, xs, dy, B
    xp = F.pad(xp, (0, 0, 0, 1))
    return xp, (0 if xs == 0 else (B + 1) * D), F.pad(dy, (0, 0, 0, 1)), B + 1


def _stacked_bias(bias, G, D):
    if bias is None:
        return None
    bias = _f32c(bias, "bias").reshape(-1)
    if bias.numel() != G * D:
        raise RuntimeError("stacked bias must have G * D elements")
    return bias


class WHVIStackedFunction(Function):
    """WHVIStackedMatrix.forward (src/weights.py:182-208) for all G blocks in one C-ABI call per direction
    (``whvi_stacked_fwd_f32`` / ``whvi_stacked_bwd_f32``): pad, reparameterisation, G x S virtual samples through the fused layer
    kernel, bias, optional ReLU, concatenation, slice.  ``params`` = G x s1, G x s2, G x g_mu, G x g_rho (the blocks' own
    parameters, so autograd routes the gradients); ``eps`` (G, S, D).

    A bfloat16 ``x`` runs the bf16 twins (``whvi_stacked_fwd_bf16`` / ``whvi_stacked_bwd_bf16``): y and dx are bf16, the fp32
    calls on the widened inputs rounded once; the parameter gradients are fp32 and bit-identical to the fp32 calls'."""

    @staticmethod
    def forward(ctx, x, eps, bias, n_out, relu_out, relu_in, *params):
        G = len(params) // 4
        eps = _f32c(eps, "eps")
        _, S, D = eps.shape
        x = _act(x, "x")
        name = "whvi_stacked_fwd_bf16" if x.dtype == torch.bfloat16 else "whvi_stacked_fwd_f32"
        n_in = x.size(-1)
        lib = _lib.lib()
        dev = x.device
        st = _stream(dev)
        with torch.cuda.device(dev):
            xp, B, xs = _stacked_input(x, S, D)
            (s1p, s2p, mup, rhop), stride = _stacked_vectors([params[i * G:(i + 1) * G] for i in range(4)], D)
            bias = _stacked_bias(bias, G, D)
            g = torch.empty((G, S, D), dtype=torch.float32, device=dev)
            yb = torch.empty((G, S, B, D), dtype=x.dtype, device=dev)
            y = torch.empty((S, B, n_out), dtype=x.dtype, device=dev)
            with _Timed(name):
                rc = getattr(lib, name)(xp.data_ptr(), xs, mup.data_ptr(), rhop.data_ptr(), s1p.data_ptr(), s2p.data_ptr(), stride,
                                        eps.data_ptr(), _ptr(bias), g.data_ptr(), yb.data_ptr(), y.data_ptr(), S, B, D, G, n_out,
                                        1 if relu_out else 0, st)
            _lib.check(rc, name)
        ctx.save_for_backward(xp, eps, g, s1p, s2p, rhop)
        ctx.meta = (S, B, D, G, xs, n_in, n_out, stride, bool(relu_in), bias is not None, x.dim())
        return y

    @staticmethod
    def backward(ctx, dy):
        xp, eps, g, s1p, s2p, rhop = ctx.saved_tensors
        S, B, D, G, xs, n_in, n_out, stride, relu_in, has_bias, xdim = ctx.meta
        bf16 = xp.dtype == torch.bfloat16
        dy = _bf16c(dy, "dy") if bf16 else _f32c(dy, "dy")
        name = "whvi_stacked_bwd_bf16" if bf16 else "whvi_stacked_bwd_f32"
        dev = dy.device
        lib = _lib.lib()
        want_dx = ctx.needs_input_grad[0]
        xp, xs, dy, Bc = _stacked_bwd_rows(xp, xs, dy, B, D)
        with torch.cuda.device(dev):
            ws = _workspace(dev, _query("whvi_stacked_bwd_workspace_bytes", S, Bc, D, G, 1 if want_dx else 0)[0])
            out = torch.empty((5 if has_bias else 4, G, D), dtype=torch.float32, device=dev)   # dmu, drho, ds1, ds2, [dbias]
            dx = torch.empty((S, Bc, n_in), dtype=xp.dtype, device=dev) if want_dx else None
            with _Timed(name):
                rc = getattr(lib, name)(xp.data_ptr(), xs, dy.data_ptr(), g.data_ptr(), rhop.data_ptr(), s1p.data_ptr(), s2p.data_ptr(),
                                        stride, eps.data_ptr(), _ptr(dx), n_in, out[0].data_ptr(), out[1].data_ptr(),
                                        out[2].data_ptr(), out[3].data_ptr(), out[4].data_ptr() if has_bias else None,
                                        ws.data_ptr(), ws.numel(), S, Bc, D, G, n_out, 1 if relu_in else 0, _stream(dev))
            _lib.check(rc, name)
        if want_dx and Bc != B:
            dx = dx[:, :B]
        if want_dx and xdim == 2:
            dx = dx.sum(dim=0)
        dbias = out[4].reshape(1, G * D) if has_bias and ctx.needs_input_grad[2] else None
        grads = [out[2, k] for k in range(G)] + [out[3, k] for k in range(G)] + [out[0, k] for k in range(G)] + [out[1, k] for k in range(G)]
        return (dx, None, dbias, None, None, None, *grads)


def whvi_stacked(x, eps, bias, n_out, blocks_s1, blocks_s2, blocks_mu, blocks_rho, relu_out=False, relu_in=False):
    return WHVIStackedFunction.apply(x, eps, bias, n_out, relu_out, relu_in, *blocks_s1, *blocks_s2, *blocks_mu, *blocks_rho)


class WHVIStackedGFunction(Function):
    """The Stacked layer from g (G, S, D) given, however it was drawn (``whvi_stacked_fwd_g_f32`` / ``whvi_stacked_bwd_g_f32``):
    the dense posterior's path, g from ``reparam_dense_grouped``.  ``params`` = G x s1, G x s2; the backward returns dg.  A bfloat16
    ``x`` runs the bf16 twins, as ``WHVIStackedFunction``."""

    @staticmethod
    def forward(ctx, x, g, bias, n_out, relu_out, relu_in, *params):
        G = len(params) // 2
        g = _f32c(g, "g")
        _, S, D = g.shape
        x = _act(x, "x")
        name = "whvi_stacked_fwd_g_bf16" if x.dtype == torch.bfloat16 else "whvi_stacked_fwd_g_f32"
        n_in = x.size(-1)
        dev = x.device
        with torch.cuda.device(dev):
            xp, B, xs = _stacked_input(x, S, D)
            (s1p, s2p), stride = _stacked_vectors([params[:G], params[G:]], D)
            bias = _stacked_bias(bias, G, D)
            yb = torch.empty((G, S, B, D), dtype=x.dtype, device=dev)
            y = torch.empty((S, B, n_out), dtype=x.dtype, device=dev)
            with _Timed(name):
                rc = getattr(_lib.lib(), name)(xp.data_ptr(), xs, g.data_ptr(), s1p.data_ptr(), s2p.data_ptr(), stride, _ptr(bias),
                                               yb.data_ptr(), y.data_ptr(), S, B, D, G, n_out, 1 if relu_out else 0, _stream(dev))
            _lib.check(rc, name)
        ctx.save_for_backward(xp, g, s1p, s2p)
        ctx.meta = (S, B, D, G, xs, n_in, n_out, stride, bool(relu_in), bias is not None, x.dim())
        return y

    @staticmethod
    def backward(ctx, dy):
        xp, g, s1p, s2p = ctx.saved_tensors
        S, B, D, G, xs, n_in, n_out, stride, relu_in, has_bias, xdim = ctx.meta
        bf16 = xp.dtype == torch.bfloat16
        dy = _bf16c(dy, "dy") if bf16 else _f32c(dy, "dy")
        name = "whvi_stacked_bwd_g_bf16" if bf16 else "whvi_stacked_bwd_g_f32"
        dev = dy.device
        want_dx = ctx.needs_input_grad[0]
        xp, xs, dy, Bc = _stacked_bwd_rows(xp, xs, dy, B, D)
        with torch.cuda.device(dev):
            ws = _workspace(dev, _query("whvi_stacked_bwd_workspace_bytes", S, Bc, D, G, 1 if want_dx else 0)[0])
            dg = torch.empty((G, S, D), dtype=torch.float32, device=dev)
            out = torch.empty((3 if has_bias else 2, G, D), dtype=torch.float32, device=dev)   # ds1, ds2, [dbias]
            dx = torch.empty((S, Bc, n_in), dtype=xp.dtype, device=dev) if want_dx else None
            with _Timed(name):
                rc = getattr(_lib.lib(), name)(xp.data_ptr(), xs, dy.data_ptr(), g.data_ptr(), s1p.data_ptr(), s2p.data_ptr(), stride,
                                               _ptr(dx), n_in, dg.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                                               out[2].data_ptr() if has_bias else None, ws.data_ptr(), ws.numel(), S, Bc, D, G, n_out,
                                               1 if relu_in else 0, _stream(dev))
            _lib.check(rc, name)
        if want_dx and Bc != B:
            dx = dx[:, :B]
        if want_dx and xdim == 2:
            dx = dx.sum(dim=0)
        dbias = out[2].reshape(1, G * D) if has_bias and ctx.needs_input_grad[2] else None
        return (dx, dg, dbias, None, None, None, *out[0].unbind(0), *out[1].unbind(0))


def whvi_stacked_g(x, g, bias, n_out, blocks_s1, blocks_s2, relu_out=False, relu_in=False):
    return WHVIStackedGFunction.apply(x, g, bias, n_out, relu_out, relu_in, *blocks_s1, *blocks_s2)


class WHVIColumnFunction(Function):
    """WHVIColumnMatrix.forward (src/weights.py:231-251, PAPER semantics) in one C-ABI call per direction
    (``whvi_column_fwd_f32`` / ``whvi_column_bwd_f32``): reparameterisation, ONE FWHT of g per MC sample, the 1-wide product,
    the bias.  ``x``: (B, n) / (S, B, n) when ``transposed`` (-> (S, B, 1)), (B, 1) / (S, B, 1) otherwise (-> (S, B, n)).

    A bfloat16 ``x`` runs the bf16 twins: x and dx are bf16, and so are y and dy of the plain form; the transposed form's output
    (S, B, 1) stays fp32 (``include/whvi_b200.h``).  The parameter gradients are fp32, bit-identical to the fp32 calls'."""

    @staticmethod
    def forward(ctx, x, eps, mu, rho, s1, s2, bias, n, transposed, relu_out, relu_in):
        x, eps = _act(x, "x"), _f32c(eps, "eps")
        mu, rho, s1, s2 = _f32c(mu, "g_mu"), _f32c(rho, "g_rho"), _f32c(s1, "s1"), _f32c(s2, "s2")
        S, D = eps.shape
        width = n if transposed else 1
        if x.size(-1) != width:
            raise RuntimeError(f"last dimension of x must be {width}, got {x.size(-1)}")
        if x.dim() == 2:
            B, xs = x.size(0), 0
        elif x.dim() == 3 and x.size(0) == S:
            B, xs = x.size(1), x.size(1) * width
        else:
            raise RuntimeError(f"x must be (B, {width}) or (S, B, {width}) with S = {S}; got {tuple(x.shape)}")
        if bias is not None:
            bias = _f32c(bias, "bias").reshape(-1)
        dev = x.device
        g = torch.empty((S, D), dtype=torch.float32, device=dev)
        hg = torch.empty((S, D), dtype=torch.float32, device=dev)    # H g, kept for the backward
        y = torch.empty((S, B, 1 if transposed else n), dtype=torch.float32 if transposed else x.dtype, device=dev)
        name = "whvi_column_fwd_bf16" if x.dtype == torch.bfloat16 else "whvi_column_fwd_f32"
        with torch.cuda.device(dev), _Timed(name):
            rc = getattr(_lib.lib(), name)(x.data_ptr(), xs, mu.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(), eps.data_ptr(),
                                           _ptr(bias), g.data_ptr(), hg.data_ptr(), y.data_ptr(), S, B, D, n, 1 if transposed else 0,
                                           1 if relu_out else 0, _stream(dev))
        _lib.check(rc, name)
        ctx.save_for_backward(x, eps, hg, rho, s1, s2)
        ctx.meta = (S, B, D, n, xs, bool(transposed), bool(relu_in), bias is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, eps, hg, rho, s1, s2 = ctx.saved_tensors
        S, B, D, n, xs, transposed, relu_in, has_bias = ctx.meta
        bf16 = x.dtype == torch.bfloat16
        dy = _bf16c(dy, "dy") if bf16 and not transposed else _f32c(dy, "dy")
        name = "whvi_column_bwd_bf16" if bf16 else "whvi_column_bwd_f32"
        dev = dy.device
        lib = _lib.lib()
        want_dx = ctx.needs_input_grad[0]
        with torch.cuda.device(dev):
            ws = _workspace(dev, _query("whvi_column_bwd_workspace_bytes", S, D, n)[0])
            out = torch.empty((4, D), dtype=torch.float32, device=dev)   # dmu, drho, ds1, ds2
            dbias = torch.empty((1, 1 if transposed else n), dtype=torch.float32, device=dev) if has_bias else None
            dx = torch.empty((S, B, n if transposed else 1), dtype=x.dtype, device=dev) if want_dx else None
            with _Timed(name):
                rc = getattr(lib, name)(x.data_ptr(), xs, dy.data_ptr(), hg.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(),
                                        eps.data_ptr(), _ptr(dx), out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
                                        out[3].data_ptr(), _ptr(dbias), ws.data_ptr(), ws.numel(), S, B, D, n, 1 if transposed else 0,
                                        1 if relu_in else 0, _stream(dev))
            _lib.check(rc, name)
        if want_dx and xs == 0:
            dx = dx.sum(dim=0)
        return dx, None, out[0], out[1], out[2], out[3], dbias, None, None, None, None


def whvi_column(x, eps, mu, rho, s1, s2, bias, n, transposed, relu_out=False, relu_in=False):
    return WHVIColumnFunction.apply(x, eps, mu, rho, s1, s2, bias, n, transposed, relu_out, relu_in)


class WHVIColumnGFunction(Function):
    """The Column layer from g (S, D) given, however it was drawn (``whvi_column_fwd_g_f32`` / ``whvi_column_bwd_g_f32``): the
    dense posterior's path, g from ``reparam_dense``.  The backward returns dg.  A bfloat16 ``x`` runs the bf16 twins, as
    ``WHVIColumnFunction``."""

    @staticmethod
    def forward(ctx, x, g, s1, s2, bias, n, transposed, relu_out, relu_in):
        x, g, s1, s2 = _act(x, "x"), _f32c(g, "g"), _f32c(s1, "s1"), _f32c(s2, "s2")
        S, D = g.shape
        width = n if transposed else 1
        if x.size(-1) != width:
            raise RuntimeError(f"last dimension of x must be {width}, got {x.size(-1)}")
        if x.dim() == 2:
            B, xs = x.size(0), 0
        elif x.dim() == 3 and x.size(0) == S:
            B, xs = x.size(1), x.size(1) * width
        else:
            raise RuntimeError(f"x must be (B, {width}) or (S, B, {width}) with S = {S}; got {tuple(x.shape)}")
        if bias is not None:
            bias = _f32c(bias, "bias").reshape(-1)
        dev = x.device
        hg = torch.empty((S, D), dtype=torch.float32, device=dev)
        y = torch.empty((S, B, 1 if transposed else n), dtype=torch.float32 if transposed else x.dtype, device=dev)
        name = "whvi_column_fwd_g_bf16" if x.dtype == torch.bfloat16 else "whvi_column_fwd_g_f32"
        with torch.cuda.device(dev), _Timed(name):
            rc = getattr(_lib.lib(), name)(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(bias), hg.data_ptr(),
                                           y.data_ptr(), S, B, D, n, 1 if transposed else 0, 1 if relu_out else 0, _stream(dev))
        _lib.check(rc, name)
        ctx.save_for_backward(x, hg, s1, s2)
        ctx.meta = (S, B, D, n, xs, bool(transposed), bool(relu_in), bias is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, hg, s1, s2 = ctx.saved_tensors
        S, B, D, n, xs, transposed, relu_in, has_bias = ctx.meta
        bf16 = x.dtype == torch.bfloat16
        dy = _bf16c(dy, "dy") if bf16 and not transposed else _f32c(dy, "dy")
        name = "whvi_column_bwd_g_bf16" if bf16 else "whvi_column_bwd_g_f32"
        dev = dy.device
        want_dx = ctx.needs_input_grad[0]
        with torch.cuda.device(dev):
            ws = _workspace(dev, _query("whvi_column_bwd_workspace_bytes", S, D, n)[0])
            dg = torch.empty((S, D), dtype=torch.float32, device=dev)
            out = torch.empty((2, D), dtype=torch.float32, device=dev)   # ds1, ds2
            dbias = torch.empty((1, 1 if transposed else n), dtype=torch.float32, device=dev) if has_bias else None
            dx = torch.empty((S, B, n if transposed else 1), dtype=x.dtype, device=dev) if want_dx else None
            with _Timed(name):
                rc = getattr(_lib.lib(), name)(x.data_ptr(), xs, dy.data_ptr(), hg.data_ptr(), s1.data_ptr(), s2.data_ptr(), _ptr(dx),
                                               dg.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), _ptr(dbias), ws.data_ptr(),
                                               ws.numel(), S, B, D, n, 1 if transposed else 0, 1 if relu_in else 0, _stream(dev))
            _lib.check(rc, name)
        if want_dx and xs == 0:
            dx = dx.sum(dim=0)
        return dx, dg, out[0], out[1], dbias, None, None, None, None


def whvi_column_g(x, g, s1, s2, bias, n, transposed, relu_out=False, relu_in=False):
    return WHVIColumnGFunction.apply(x, g, s1, s2, bias, n, transposed, relu_out, relu_in)


class KLGroupedFunction(Function):
    """Sum of the blocks' KL terms (src/weights.py:162-164) with all gradients in one launch."""

    @staticmethod
    def forward(ctx, lambda_, mode, *params):
        G = len(params) // 2
        mus, rhos = params[:G], params[G:]
        D = mus[0].numel()
        sm, sr = uniform_stride(mus), uniform_stride(rhos)
        if sm is None or sm != sr:
            mup, rhop, stride = torch.stack([t.detach() for t in mus]), torch.stack([t.detach() for t in rhos]), D
        else:
            mup, rhop, stride = mus[0].detach(), rhos[0].detach(), sm
        dev = mup.device
        out = torch.empty(1, dtype=torch.float32, device=dev)
        need_grad = any(ctx.needs_input_grad[2:])
        grads = torch.empty((2, G, D), dtype=torch.float32, device=dev) if need_grad else None
        with torch.cuda.device(dev), _Timed("whvi_kl_grouped_f32"):
            rc = _lib.lib().whvi_kl_grouped_f32(mup.data_ptr(), rhop.data_ptr(), float(lambda_), D, G, stride, int(mode), out.data_ptr(),
                                                grads[0].data_ptr() if need_grad else None, grads[1].data_ptr() if need_grad else None,
                                                1.0, _stream(dev))
        _lib.check(rc, "whvi_kl_grouped_f32")
        ctx.G = G
        if need_grad:
            ctx.save_for_backward(grads)
        return out.reshape(())

    @staticmethod
    def backward(ctx, dkl):
        (grads,) = ctx.saved_tensors
        gr = grads * dkl
        G = ctx.G
        return (None, None, *[gr[0, k] for k in range(G)], *[gr[1, k] for k in range(G)])


def kl_gaussian_grouped(mus, rhos, lambda_, mode=0):
    return KLGroupedFunction.apply(lambda_, mode, *mus, *rhos)


class KLFunction(Function):
    """KL(N(mu, softplus(rho)) || N(0, lambda)) value + gradient in one kernel.
    mode 0 = the reference's formula (src/utils.py:49-71), mode 1 = sigma^2 form."""

    @staticmethod
    def forward(ctx, mu, rho, lambda_, mode):
        mu, rho = _f32c(mu, "g_mu"), _f32c(rho, "g_rho")
        D = mu.numel()
        out = torch.empty(1, dtype=torch.float32, device=mu.device)
        need_grad = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        dmu = torch.empty_like(mu) if need_grad else None
        drho = torch.empty_like(rho) if need_grad else None
        with torch.cuda.device(mu.device), _Timed("whvi_kl_f32"):
            rc = _lib.lib().whvi_kl_f32(mu.data_ptr(), rho.data_ptr(), float(lambda_), D, int(mode), out.data_ptr(),
                                        _ptr(dmu), _ptr(drho), 1.0, 0, _stream(mu.device))
        _lib.check(rc, "whvi_kl_f32")
        if need_grad:
            ctx.save_for_backward(dmu, drho)
        return out.reshape(())

    @staticmethod
    def backward(ctx, dkl):
        dmu, drho = ctx.saved_tensors
        return dmu * dkl, drho * dkl, None, None


def kl_gaussian(mu, rho, lambda_, mode=0):
    return KLFunction.apply(mu, rho, lambda_, mode)


# ---------------------------------------------------------------------------------------------- categorical likelihood
def _categorical_args(logits, labels):
    """(logits, labels, S, B, K) for the categorical calls.  Shapes and dtypes are checked before the device, so every misuse
    gets its own message; nothing here reads the labels (a device sync would break CUDA-graph capture): labels outside
    [0, K) come back as NaN from the kernels."""
    if logits.dim() != 3:
        raise RuntimeError(f"logits must be (S, B, K), got {tuple(logits.shape)}")
    S, B, K = logits.shape
    if labels.dim() != 1 or labels.size(0) != B:
        raise RuntimeError(f"labels must be ({B},) for logits {tuple(logits.shape)}, got {tuple(labels.shape)}")
    if logits.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError(f"logits must be float32 or bfloat16 (got {logits.dtype})")
    if labels.dtype != torch.int64:
        raise RuntimeError(f"labels must be int64 (got {labels.dtype})")
    if logits.device.type != "cuda" or labels.device != logits.device:
        raise RuntimeError("logits and labels must be CUDA tensors on one device")
    return logits.contiguous(), labels.contiguous(), S, B, K


class CategoricalNLLFunction(Function):
    """sum_{s,b} -log softmax(z[s, b])[y_b] for (S, B, K) logits (fp32 or bf16) and (B,) int64 labels, as a 0-d fp32 tensor
    (``whvi_categorical_nll_*``: max-subtracted log-sum-exp per row, fixed-order fp64 reduction).  The backward is
    ``whvi_categorical_nll_bwd_*`` with the incoming gradient read from the device (no sync, graph-capturable); dz has the
    logits' dtype."""

    @staticmethod
    def forward(ctx, logits, labels):
        logits, labels, S, B, K = _categorical_args(logits, labels)
        bf16 = logits.dtype == torch.bfloat16
        name = "whvi_categorical_nll_bf16" if bf16 else "whvi_categorical_nll_f32"
        dev = logits.device
        want_grad = ctx.needs_input_grad[0]
        lse = torch.empty((S, B), dtype=torch.float32, device=dev) if want_grad else None
        total = torch.empty(1, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            ws = _workspace(dev, _query("whvi_categorical_sizes", S * B, K)[0])
            with _Timed(name, f"K={K}"):
                rc = getattr(_lib.lib(), name)(logits.data_ptr(), labels.data_ptr(), _ptr(lse), total.data_ptr(), ws.data_ptr(), ws.numel(),
                                               S, B, K, _stream(dev))
        _lib.check(rc, name)
        if want_grad:
            ctx.save_for_backward(logits, labels, lse)
        return total.reshape(())

    @staticmethod
    def backward(ctx, d_total):
        logits, labels, lse = ctx.saved_tensors
        S, B, K = logits.shape
        c = _f32c(d_total, "grad_output").reshape(1)
        dz = torch.empty_like(logits)
        name = "whvi_categorical_nll_bwd_bf16" if logits.dtype == torch.bfloat16 else "whvi_categorical_nll_bwd_f32"
        with torch.cuda.device(logits.device), _Timed(name, f"K={K}"):
            rc = getattr(_lib.lib(), name)(logits.data_ptr(), labels.data_ptr(), lse.data_ptr(), c.data_ptr(), dz.data_ptr(), S, B, K,
                                           _stream(logits.device))
        _lib.check(rc, name)
        return dz, None


def categorical_nll(logits, labels):
    return CategoricalNLLFunction.apply(logits, labels)


def categorical_predictive_(logits, labels, prob_sum, loglik_sum=None, accumulate=False):
    """prob_sum (+)= sum_s softmax(logits[s]) (B, K) and, with ``labels``, loglik_sum (+)= sum_s log softmax(logits[s])[labels]
    (B,), samples ascending (``whvi_categorical_predictive_*``).  ``logits`` (S, B, K) fp32 or bf16 may be a sample-slice of a
    larger tensor (rows contiguous, any sample stride); ``accumulate`` continues the sums of earlier sample chunks in the order
    of one call over all samples, so chunked evaluation gives the same bits.  No autograd."""
    if logits.dim() != 3:
        raise RuntimeError(f"logits must be (S, B, K), got {tuple(logits.shape)}")
    S, B, K = logits.shape
    if labels is not None:
        labels = _categorical_args(logits[:0], labels)[1]
    elif logits.dtype not in (torch.float32, torch.bfloat16) or logits.device.type != "cuda":
        raise RuntimeError("logits must be a float32 or bfloat16 CUDA tensor")
    if (labels is None) != (loglik_sum is None):
        raise RuntimeError("labels and loglik_sum go together")
    if logits.stride(2) != 1 or logits.stride(1) != K:
        logits = logits.contiguous()
    stride = logits.stride(0) if S > 1 else B * K
    for t, name, n in ((prob_sum, "prob_sum", B * K), (loglik_sum, "loglik_sum", B)):
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n or t.device != logits.device):
            raise RuntimeError(f"{name} must be a contiguous float32 tensor with {n} elements on {logits.device}")
    name = "whvi_categorical_predictive_bf16" if logits.dtype == torch.bfloat16 else "whvi_categorical_predictive_f32"
    with torch.cuda.device(logits.device), _Timed(name, f"K={K}"):
        rc = getattr(_lib.lib(), name)(logits.data_ptr(), stride, _ptr(labels), prob_sum.data_ptr(), _ptr(loglik_sum), S, B, K,
                                       1 if accumulate else 0, _stream(logits.device))
    _lib.check(rc, name)
    return prob_sum, loglik_sum


# ---------------------------------------------------------------------------------------------- convolution patches
def conv_output_size(n: int, k: int, stride: int, pad: int, dil: int) -> int:
    """Output length of a convolution along one spatial axis (torch.nn.Conv2d's formula, floor)."""
    return (n + 2 * pad - dil * (k - 1) - 1) // stride + 1


def _image_dims(x):
    """(S or None, B, H, W, C, x_sample_stride) of a channels-last (B, H, W, C) or (S, B, H, W, C) image batch."""
    if x.dim() == 4:
        return (None, *x.shape, 0)
    if x.dim() == 5:
        return (x.size(0), *x.shape[1:], x[0].numel())
    raise RuntimeError(f"images must be (B, H, W, C) or (S, B, H, W, C) channels-last, got {tuple(x.shape)}")


def im2col_(x, geom, ld):
    """Patch matrix of a channels-last image batch (``whvi_im2col_*``): ``x`` (B, H, W, C) -> (B Ho Wo, ld), or (S, B, H, W, C)
    -> (S, B Ho Wo, ld), fp32 or bf16 as ``x``.  ``geom`` = (kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w).  Column
    (i kw + j) C + c holds tap (i, j) of channel c; columns from C kh kw to ld - 1 are zero.  No autograd."""
    x = _act(x, "x")
    S, B, H, W, C, xs = _image_dims(x)
    kh, kw, sh, sw, ph, pw, dh, dw = geom
    Ho, Wo = conv_output_size(H, kh, sh, ph, dh), conv_output_size(W, kw, sw, pw, dw)
    out = torch.empty(((B * Ho * Wo, ld) if S is None else (S, B * Ho * Wo, ld)), dtype=x.dtype, device=x.device)
    name = "whvi_im2col_bf16" if x.dtype == torch.bfloat16 else "whvi_im2col_f32"
    with torch.cuda.device(x.device), _Timed(name):
        rc = getattr(_lib.lib(), name)(x.data_ptr(), xs, out.data_ptr(), 1 if S is None else S, B, H, W, C, *geom, ld, _stream(x.device))
    _lib.check(rc, name)
    return out


def col2im_(dpatches, geom, image_shape, sum_samples=False):
    """Adjoint of ``im2col_`` (``whvi_col2im_*``): the (B Ho Wo, ld) or (S, B Ho Wo, ld) patch gradient scattered back to the
    channels-last image of ``image_shape`` (B, H, W, C), each input element summing its taps i ascending, j ascending in fp32.
    ``sum_samples``: a (S, B Ho Wo, ld) gradient is reduced over s ascending into one (B, H, W, C) block, the gradient of an
    input shared by the samples; otherwise the result has the sample axis of ``dpatches``.  No autograd."""
    dp = _act(dpatches, "dpatches")
    B, H, W, C = image_shape
    S = 1 if dp.dim() == 2 else dp.size(0)
    ld = dp.size(-1)
    shape = (B, H, W, C) if dp.dim() == 2 or sum_samples else (S, B, H, W, C)
    dx = torch.empty(shape, dtype=dp.dtype, device=dp.device)
    name = "whvi_col2im_bf16" if dp.dtype == torch.bfloat16 else "whvi_col2im_f32"
    with torch.cuda.device(dp.device), _Timed(name):
        rc = getattr(_lib.lib(), name)(dp.data_ptr(), ld, dx.data_ptr(), S, B, H, W, C, *geom, 1 if sum_samples else 0, _stream(dp.device))
    _lib.check(rc, name)
    return dx


class Im2ColFunction(Function):
    """``im2col_`` with its adjoint as the backward: the patch gather of ``WHVIConv2d``.  A layer call on the patch matrix
    follows it, and autograd composes the two, so every parameter gradient comes from the layer's own kernels.  For an input
    shared by the samples the patches are one (B Ho Wo, ld) block, which the layer reads for every sample and whose gradient
    it returns already summed over the samples; col2im then scatters that one block.  The backward is skipped when ``x``
    needs no gradient."""

    @staticmethod
    def forward(ctx, x, geom, ld):
        ctx.geom, ctx.image_shape = geom, tuple(x.shape[-4:])
        return im2col_(x, geom, ld)

    @staticmethod
    def backward(ctx, dpatches):
        if not ctx.needs_input_grad[0]:
            return None, None, None
        return col2im_(dpatches, ctx.geom, ctx.image_shape), None, None


def im2col(x, geom, ld):
    return Im2ColFunction.apply(x, geom, ld)
