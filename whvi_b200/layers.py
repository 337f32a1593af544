"""``WHVILinear``: the reference's shape dispatcher (``src/layers.py:19-48``) over the
B200-native weight modules."""
from __future__ import annotations

import torch.nn as nn

from .weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix


class WHVI:
    """Marker base for layers that carry a KL term (``src/layers.py:7-16``)."""

    @property
    def kl(self):
        return 0.0


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
        kw = dict(lambda_=lambda_, bias=bias, semantics=semantics, kl_mode=kl_mode, covariance=covariance)
        if n_in == 1:
            self.weight_submodule = WHVIColumnMatrix(n_out, **kw)
        elif n_out == 1:
            self.weight_submodule = WHVIColumnMatrix(n_in, transposed=True, **kw)
        elif n_in == n_out and n_in & (n_in - 1) == 0:
            self.weight_submodule = WHVISquarePow2Matrix(n_in, **kw)
        else:
            self.weight_submodule = WHVIStackedMatrix(n_in, n_out, **kw)

    @property
    def mc_samples(self):
        return self.weight_submodule.mc_samples

    @mc_samples.setter
    def mc_samples(self, value):
        self.weight_submodule.mc_samples = value

    def square_blocks(self):
        """Every WHVISquarePow2Matrix of this layer in the reference's draw order."""
        w = self.weight_submodule
        if isinstance(w, WHVISquarePow2Matrix):
            return [w]
        if isinstance(w, WHVIStackedMatrix):
            return list(w.weight_matrices)
        return [w.weight_submodule]

    @property
    def kl(self):
        """KL divergence from the prior to the variational posterior."""
        return self.weight_submodule.kl

    def forward(self, x):
        return self.weight_submodule.forward(x)
