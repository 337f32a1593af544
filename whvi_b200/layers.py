"""``WHVILinear``: the reference's shape dispatcher (``src/layers.py:19-48``) over the
B200-native weight modules; ``WHVIConv2d``: the same weights as a convolution's filter bank."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import functional as WF
from .weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix


class WHVI:
    """Marker base for layers that carry a KL term (``src/layers.py:7-16``)."""

    @property
    def kl(self):
        return 0.0


def _weight_module(n_in, n_out, **kw):
    """The weight module of an n_in -> n_out WHVI map: Column for a 1-wide side, square for equal powers of two, else Stacked."""
    if n_in == 1:
        return WHVIColumnMatrix(n_out, **kw)
    if n_out == 1:
        return WHVIColumnMatrix(n_in, transposed=True, **kw)
    if n_in == n_out and n_in & (n_in - 1) == 0:
        return WHVISquarePow2Matrix(n_in, **kw)
    return WHVIStackedMatrix(n_in, n_out, **kw)


def _square_blocks(w):
    if isinstance(w, WHVISquarePow2Matrix):
        return [w]
    if isinstance(w, WHVIStackedMatrix):
        return list(w.weight_matrices)
    return [w.weight_submodule]


class WHVILinear(nn.Module, WHVI):
    def __init__(self, n_in, n_out, lambda_=1e-5, bias=False, *, semantics="paper", kl_mode=0, covariance="diag"):
        """WHVI feed-forward layer.

        :param int n_in: input dimensionality.
        :param int n_out: output dimensionality.
        :param float lambda_: prior variance.
        :param boolean bias: add an optimised (non-variational) bias after the linear map.
        :param str semantics: "paper" | "reference", see ``whvi_b200.weights``.
        :param str covariance: "diag" (the reference's posterior) | "dense" (g = mu + L eps with a lower-triangular L per
            square block, the paper's full-covariance posterior; PAPER semantics), see ``WHVISquarePow2Matrix``.
        """
        super().__init__()
        self.weight_submodule = _weight_module(n_in, n_out, lambda_=lambda_, bias=bias, semantics=semantics, kl_mode=kl_mode,
                                               covariance=covariance)

    @property
    def mc_samples(self):
        return self.weight_submodule.mc_samples

    @mc_samples.setter
    def mc_samples(self, value):
        self.weight_submodule.mc_samples = value

    def square_blocks(self):
        """Every WHVISquarePow2Matrix of this layer in the reference's draw order."""
        return _square_blocks(self.weight_submodule)

    @property
    def kl(self):
        """KL divergence from the prior to the variational posterior."""
        return self.weight_submodule.kl

    def forward(self, x):
        return self.weight_submodule.forward(x)


def _pair(v, name):
    t = (v, v) if isinstance(v, int) else tuple(v)
    if len(t) != 2 or not all(isinstance(e, int) for e in t):
        raise ValueError(f"{name} must be an int or a pair of ints, got {v!r}")
    return t


class WHVIConv2d(nn.Module, WHVI):
    """2-D convolution whose filter bank is a WHVI weight: the ``C_out x (C_in kh kw)`` matrix W = S1 H diag(g) H S2 of
    ``WHVILinear(C_in kh kw, C_out)``, applied to every patch of the input.

    Column order: tap (i, j) of input channel c is column (i kw + j) C_in + c of W (channels fastest), so the equivalent torch
    filter is ``W.reshape(C_out, kh, kw, C_in).permute(0, 3, 1, 2)`` (``sample_filters`` returns it).

    The forward is a patch gather (``functional.im2col``: the ``whvi_im2col_*`` kernels on the channels-last image) followed by
    the layer call of the weight module on the (S|1, B Ho Wo, ld) patch matrix, rows in (b, oh, ow) order; the backward is the
    layer's backward and the patch scatter (``whvi_col2im_*``).  ``ld`` is the block width D_in for square and Stacked weights,
    so the patches are that call's zero-padded input as they are, and C_in kh kw for Column weights.

    Input: ``(B, C_in, H, W)``, shared by all MC samples, or ``(S, B, C_in, H, W)``, float32 or bfloat16 (bf16 activations, as
    ``WHVILinear``), on CUDA.  Output: ``(S, B, C_out, Ho, Wo)`` as a view of the contiguous ``(S, B, Ho, Wo, C_out)`` layer output,
    so each (s, b) image is ``torch.channels_last`` and merging S and B for foreign modules (pooling, ReLU) is a view; a
    channels_last input costs no copy.  Standalone, with ``mc_samples`` unset, a 4-D input gets one draw and a 4-D output, as
    ``WHVILinear`` does for 2-D inputs.  A single output channel runs the transposed Column weight, whose output stays fp32.

    ``state_dict`` keys and the initial values (same RNG draws in the same order) are those of ``WHVILinear(C_in kh kw, C_out)``.
    PAPER semantics only: the reference has no convolution, and its as-written semantics collapse W to a diagonal."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, lambda_=1e-5, bias=False, *,
                 kl_mode=0, covariance="diag", semantics="paper"):
        if semantics != "paper":
            raise ValueError('WHVIConv2d implements semantics="paper" only (the reference has no convolution, and its '
                             'as-written semantics collapse W to a diagonal)')
        super().__init__()
        self.in_channels, self.out_channels = int(in_channels), int(out_channels)
        if self.in_channels < 1 or self.out_channels < 1:
            raise ValueError("in_channels and out_channels must be positive")
        self.kernel_size = _pair(kernel_size, "kernel_size")
        self.stride = _pair(stride, "stride")
        self.padding = _pair(padding, "padding")
        self.dilation = _pair(dilation, "dilation")
        if min(self.kernel_size + self.stride + self.dilation) < 1 or min(self.padding) < 0:
            raise ValueError("kernel_size, stride and dilation must be positive, padding non-negative")
        kh, kw = self.kernel_size
        self.n_in = self.in_channels * kh * kw
        self.weight_submodule = _weight_module(self.n_in, self.out_channels, lambda_=lambda_, bias=bias, semantics="paper",
                                               kl_mode=kl_mode, covariance=covariance)
        w = self.weight_submodule
        self.ld = w.D_in if isinstance(w, WHVIStackedMatrix) else (w.D if isinstance(w, WHVISquarePow2Matrix) else self.n_in)

    @property
    def geometry(self):
        """(kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w), the argument order of the patch kernels."""
        return (*self.kernel_size, *self.stride, *self.padding, *self.dilation)

    def output_size(self, H, W):
        """(Ho, Wo) for an H x W input (torch.nn.Conv2d's arithmetic)."""
        kh, kw, sh, sw, ph, pw, dh, dw = self.geometry
        return WF.conv_output_size(H, kh, sh, ph, dh), WF.conv_output_size(W, kw, sw, pw, dw)

    @property
    def mc_samples(self):
        return self.weight_submodule.mc_samples

    @mc_samples.setter
    def mc_samples(self, value):
        self.weight_submodule.mc_samples = value

    def square_blocks(self):
        """Every WHVISquarePow2Matrix of this layer in the reference's draw order."""
        return _square_blocks(self.weight_submodule)

    @property
    def kl(self):
        """KL divergence from the prior to the variational posterior."""
        return self.weight_submodule.kl

    def forward(self, x):
        if x.dim() not in (4, 5) or x.size(-3) != self.in_channels:
            raise RuntimeError(f"WHVIConv2d: input must be (B, {self.in_channels}, H, W) or (S, B, {self.in_channels}, H, W), "
                               f"got {tuple(x.shape)}")
        if x.device.type != "cuda":
            raise RuntimeError("whvi_b200 runs on CUDA only (no CPU fallback); move the module and its inputs to a GPU")
        Ho, Wo = self.output_size(x.size(-2), x.size(-1))
        if Ho < 1 or Wo < 1:
            raise RuntimeError(f"WHVIConv2d: a {tuple(x.shape[-2:])} input is smaller than the dilated kernel")
        patches = WF.im2col(x.movedim(-3, -1), self.geometry, self.ld)
        y = self.weight_submodule(patches).contiguous()      # (S, B Ho Wo, C_out), or (B Ho Wo, C_out) for one standalone draw
        B = x.size(-4)
        return y.view(*y.shape[:-2], B, Ho, Wo, self.out_channels).movedim(-1, -3)

    def sample_filters(self, n_samples=None, eps=None):
        """(S, C_out, C_in, kh, kw) torch-order filters W_s for S posterior draws (the bias is not part of them): the layer call
        on the identity patch matrix
        (rows e_j zero-padded to ld), so the filters are exactly what the forward applies.  ``eps``: the draws' noise, one
        (S, D) tensor per square block in ``square_blocks()`` order (injected like ``inject_eps``); otherwise ``n_samples``
        (default: ``mc_samples``, else 1) fresh draws.  Runs under the caller's grad mode."""
        blocks = self.square_blocks()
        if eps is not None:
            eps = list(eps)
            if len(eps) != len(blocks):
                raise ValueError(f"eps needs one tensor per square block ({len(blocks)}), got {len(eps)}")
            for b, e in zip(blocks, eps):
                b.inject_eps(e)
            S = eps[0].reshape(-1, blocks[0].D).size(0)
        else:
            S = int(n_samples or self.mc_samples or 1)
        eye = torch.eye(self.n_in, self.ld, device=blocks[0].g_mu.device)
        w = self.weight_submodule
        saved, bias = self.mc_samples, w.bias
        self.mc_samples, w.bias = S, None                     # the filters alone, without the bias
        try:
            y = w(eye)                                        # (S, n_in, C_out): row j is column j of W_s
        finally:
            self.mc_samples, w.bias = saved, bias
        kh, kw = self.kernel_size
        return y.transpose(1, 2).reshape(S, self.out_channels, kh, kw, self.in_channels).permute(0, 1, 4, 2, 3)
