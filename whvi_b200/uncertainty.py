"""Predictive uncertainty of WHVI networks, computed in fp64 from the Monte Carlo sums that the kernels reduce.

Classifiers (``WHVIClassification.predictive_uncertainty`` / ``predictive_metrics``, ``distributed.reduce_predictive_uncertainty``):
the sums of ``functional.categorical_uncertainty_`` -- sum_s softmax(z_s), sum_s H[softmax(z_s)] and log sum_s p_s(y) -- give
the entropy of the MC-mean prediction, the expected entropy, their difference (the mutual information between the label and
the weights, "BALD") and the log predictive likelihood; ``brier_score`` and ``expected_calibration_error`` score the mean
prediction.  Regressors (``WHVIRegression.predictive_uncertainty``): the MC mean, its variance over the samples and the
likelihood's noise variance.  Everything here is O(B K) and runs on the sums, never on the (S, B, K) logits.
"""
from __future__ import annotations

import math
from typing import NamedTuple, Optional

import torch


class CategoricalUncertainty(NamedTuple):
    probs: torch.Tensor                     # MC-mean probabilities prob_sum / S, (B, K) fp32: what predict_proba returns
    predictive_entropy: torch.Tensor        # H[probs] (B,) fp64, total uncertainty
    expected_entropy: torch.Tensor          # (1/S) sum_s H[softmax(z_s)] (B,) fp64, aleatoric part
    mutual_information: torch.Tensor        # predictive - expected entropy (B,) fp64, epistemic part (not clamped)
    log_predictive: Optional[torch.Tensor]  # log (1/S) sum_s p_s(y) (B,) fp64, None without labels
    S: int


class RegressionUncertainty(NamedTuple):
    mean: torch.Tensor                # (1/S) sum_s y_hat_s (B, out) fp64
    epistemic_variance: torch.Tensor  # Var_s y_hat_s (B, out) fp64, the biased (1/S) variance over the samples
    aleatoric_variance: torch.Tensor  # sigma^2 of the Gaussian likelihood, broadcast to (B, out) fp64
    S: int


def categorical_uncertainty(prob_sum: torch.Tensor, ent_sum: torch.Tensor, logpred: torch.Tensor | None, S: int
                            ) -> CategoricalUncertainty:
    """The decomposition from the sums over S samples: prob_sum (B, K), ent_sum (B,) and logpred = log sum_s p_s(y) (B,) or
    None.  H[p] is computed in fp64 with 0 log 0 = 0.  The mutual information is returned as computed: when the samples agree
    it is the difference of two equal entropies, each carrying the fp32 rounding of its sums, so it can come out below zero
    by about 1e-6 log K."""
    if S < 1:
        raise ValueError("the uncertainty needs S >= 1 samples")
    probs = prob_sum / S
    p = prob_sum.to(torch.float64) / S
    predictive = -torch.special.xlogy(p, p).sum(-1)
    expected = ent_sum.to(torch.float64) / S
    log_predictive = None if logpred is None else logpred.to(torch.float64) - math.log(S)
    return CategoricalUncertainty(probs, predictive, expected, predictive - expected, log_predictive, S)


def brier_score(probs: torch.Tensor, labels: torch.Tensor) -> float:
    """mean_b sum_k (probs[b, k] - [k = labels[b]])^2, in fp64."""
    p = probs.to(torch.float64)
    onehot = torch.nn.functional.one_hot(labels, p.size(-1)).to(torch.float64)
    return float((p - onehot).square().sum(-1).mean())


def expected_calibration_error(probs: torch.Tensor, labels: torch.Tensor, n_bins: int = 15) -> float:
    """sum_bins (n_bin / B) |accuracy_bin - mean confidence_bin| over n_bins equal-width bins (i / n, (i + 1) / n] of the
    confidence max_k probs[b, k] (a confidence of 0 goes to the first bin), in fp64."""
    if n_bins < 1:
        raise ValueError("n_bins must be >= 1")
    conf, pred = probs.to(torch.float64).max(-1)
    gap = (pred == labels).to(torch.float64) - conf
    idx = torch.ceil(conf * n_bins).long().clamp(1, n_bins) - 1
    per_bin = torch.zeros(n_bins, dtype=torch.float64, device=conf.device).index_add_(0, idx, gap)
    return float(per_bin.abs().sum() / conf.numel())
