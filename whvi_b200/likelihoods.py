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
    reduced by the ``whvi_categorical_nll`` kernels.

    The options of ``torch.nn.functional.cross_entropy``, for training:
      * ``weight`` (K,): class weights w, for imbalanced data.  Kept as a non-persistent buffer, so it follows ``.to()`` /
        ``.cuda()`` and the ``state_dict`` has the same keys with and without it.
      * ``label_smoothing`` eps in [0, 1]: the target is (1 - eps) onehot(y) + eps / K.
      * ``ignore_index``: rows labelled with it add nothing to the loss or its gradient (unlabelled or padding rows, a
        "void" class).  It may lie outside [0, K), e.g. -100; any other label outside [0, K) still gives NaN.
    The row term is then ``cross_entropy(z, y, weight, ignore_index=..., label_smoothing=eps, reduction="sum")``, computed by
    the ``whvi_categorical_nll_ex`` kernels, and the estimator stays n/(m*n_mc) * sum over rows, with ignored rows counted in
    m: it is an unbiased estimate of the weighted, smoothed negative log-likelihood summed over the labelled points of a data
    set of n points.  With every option at its default the plain kernels run, as before."""

    def __init__(self, weight=None, label_smoothing: float = 0.0, ignore_index: int | None = None):
        super().__init__()
        if weight is not None:
            weight = torch.as_tensor(weight).detach().to(torch.float32).contiguous()
            if weight.dim() != 1 or weight.numel() < 2:
                raise ValueError(f"weight must be a (K,) tensor with K >= 2 (got shape {tuple(weight.shape)})")
            if not bool(torch.isfinite(weight).all()) or bool((weight < 0).any()):
                raise ValueError("weight must be finite and >= 0")
        ls = float(label_smoothing)
        if not 0.0 <= ls <= 1.0:
            raise ValueError(f"label_smoothing must be in [0, 1] (got {label_smoothing})")
        if ignore_index is not None and (isinstance(ignore_index, bool) or int(ignore_index) != ignore_index):
            raise ValueError(f"ignore_index must be an int or None (got {ignore_index!r})")
        self.register_buffer("weight", weight, persistent=False)
        self.label_smoothing = ls
        self.ignore_index = None if ignore_index is None else int(ignore_index)

    def mnll_batch_estimate(self, y: torch.Tensor, y_hat: torch.Tensor, n: int) -> torch.Tensor:
        """:param y: labels (m,) int64;  :param y_hat: logits (m, K, n_mc) as ``WHVINetwork.forward`` returns them;
        :param int n: data-set size."""
        return self.mnll_from_logits(y, y_hat.permute(2, 0, 1), n)

    def mnll_from_logits(self, y: torch.Tensor, logits: torch.Tensor, n: int) -> torch.Tensor:
        """The same estimator on sample-major (n_mc, m, K) logits, as the network produces them (no permute copy)."""
        n_mc, m, _ = logits.shape
        return (n / (m * n_mc)) * WF.categorical_nll(logits, y, self.weight, self.label_smoothing, self.ignore_index)

    def labelled(self, y: torch.Tensor) -> torch.Tensor | None:
        """Boolean mask of the rows of labels y that are not ``ignore_index``, or None without one."""
        return None if self.ignore_index is None else y != self.ignore_index

    def extra_repr(self) -> str:
        return (f"weight={'None' if self.weight is None else tuple(self.weight.shape)}, label_smoothing={self.label_smoothing}, "
                f"ignore_index={self.ignore_index}")
