"""Likelihoods (reference ``src/likelihoods.py``)."""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from . import functional as WF


class Likelihood:
    def mnll_batch_estimate(self, *args, **kwargs):
        return 0.0


class GaussianLikelihood(nn.Module, Likelihood):
    def __init__(self, sigma: float = 1.0):
        super().__init__()
        self.sigma = nn.Parameter(torch.tensor(sigma))

    def mnll_batch_estimate(self, y: torch.Tensor, y_hat: torch.Tensor, n: int) -> torch.Tensor:
        """-n/(m*n_mc) * sum_{b,i,s} log N(y[b,i] | y_hat[b,i,s], sigma)
        (``src/likelihoods.py:18-29``), as one closed-form reduction instead of a Python loop
        over outputs building ``Normal`` objects.

        :param y: targets (m, n_out);  :param y_hat: predictions (m, n_out, n_mc);
        :param int n: data-set size.
        """
        m, n_out, n_mc = y_hat.size()
        sq = (y.reshape(m, n_out, 1) - y_hat).square().sum()
        return self.mnll_from_sq_error(sq, m, n_out, n_mc, n)

    def mnll_from_sq_error(self, sq: torch.Tensor, m: int, n_out: int, n_mc: int, n: int) -> torch.Tensor:
        """The same estimator given sum_{b,i,s} (y - y_hat)^2 (which the fused last-layer
        kernel reduces on the fly)."""
        count = m * n_out * n_mc
        log_prob_sum = -count * (torch.log(self.sigma) + 0.5 * math.log(2.0 * math.pi)) - 0.5 * sq / self.sigma ** 2
        return -n / (m * n_mc) * log_prob_sum


class CategoricalLikelihood(nn.Module, Likelihood):
    """Softmax likelihood of a classifier: p(y | z) = softmax(z)[y] for the network's logits z (not in the reference, whose
    networks only regress).  No parameters.  The estimator is the Gaussian's: -n/(m*n_mc) * sum_{b,s} log p(y_b | z_{b,s}),
    reduced by the ``whvi_categorical_nll`` kernels."""

    def mnll_batch_estimate(self, y: torch.Tensor, y_hat: torch.Tensor, n: int) -> torch.Tensor:
        """:param y: labels (m,) int64;  :param y_hat: logits (m, K, n_mc) as ``WHVINetwork.forward`` returns them;
        :param int n: data-set size."""
        return self.mnll_from_logits(y, y_hat.permute(2, 0, 1), n)

    def mnll_from_logits(self, y: torch.Tensor, logits: torch.Tensor, n: int) -> torch.Tensor:
        """The same estimator on sample-major (n_mc, m, K) logits, as the network produces them (no permute copy)."""
        n_mc, m, _ = logits.shape
        return (n / (m * n_mc)) * WF.categorical_nll(logits, y)
