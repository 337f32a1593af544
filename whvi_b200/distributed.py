"""Multi-GPU plumbing for the WHVI hot path: one process per GPU (``torchrun``), MC samples
sharded across ranks, ONE flat all-reduce of the parameter gradients per step.

Every (sample, row) pair is independent given replicated parameters (SURVEY 8e), so the data
path needs no collective; the only exchange is the sum of the small parameter gradients
({d mu, d rho, d s1, d s2, d bias} of every layer plus the likelihood's sigma): 4.D floats per
square block, ~49 K floats (196 KB) for the 3 x 4096 network -- latency-bound, one NCCL call.

Scaling convention (``rank_loss``): each rank computes ``loss_r = mnll_r * n_local / S + kl / world``
on its own sample shard (``mnll_r`` already divides by its LOCAL sample count ``n_local``), so the SUM
over ranks of the gradients equals the single-process gradient of ``mean_s mnll + kl`` for even and
uneven shards alike; with ``S % world == 0`` this is the familiar ``(mnll_r + kl) / world``.

The exchange itself is ``whvi_b200.optim.FlatParams.all_reduce`` (gradients live as views of one buffer:
one NCCL call, no pack / unpack kernels); ``FlatGradAllReduce`` is the copying variant for models whose
``.grad`` tensors are managed by someone else.
"""
from __future__ import annotations

from typing import Iterable, List, Tuple

import torch
import torch.distributed as dist


def shard_samples(total_samples: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(first_sample, n_local) for this rank; samples are split as evenly as possible."""
    if total_samples < 0 or world_size < 1 or not 0 <= rank < world_size:
        raise ValueError("bad shard arguments")
    base, extra = divmod(total_samples, world_size)
    n_local = base + (1 if rank < extra else 0)
    first = rank * base + min(rank, extra)
    return first, n_local


def shard_rows(total_rows: int, rank: int, world_size: int) -> Tuple[int, int]:
    """(first_row, n_local): evaluation can shard minibatch rows instead of samples."""
    return shard_samples(total_rows, rank, world_size)


def rank_loss(mnll_local, kl, n_local: int, total_samples: int, world_size: int):
    """This rank's share of the ELBO loss such that the SUM over ranks has the gradient of
    ``mean over all S samples of mnll + kl`` (KL is replicated: every rank adds 1/world of it).
    ``mnll_local`` is the MNLL estimate over this rank's ``n_local`` samples."""
    if total_samples <= 0 or world_size < 1:
        raise ValueError("bad rank_loss arguments")
    return mnll_local * (float(n_local) / float(total_samples)) + kl * (1.0 / world_size)


class FlatGradAllReduce:
    """Sum the gradients of ``params`` across ranks through one contiguous fp32 buffer."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        self.numel = sum(p.numel() for p in self.params)
        self._flat = None

    def __call__(self, group=None) -> None:
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        if not self.params:
            return
        dev = self.params[0].device
        if self._flat is None or self._flat.device != dev:
            self._flat = torch.empty(self.numel, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:
            n = p.numel()
            if p.grad is None:
                self._flat[off:off + n].zero_()
            else:
                self._flat[off:off + n].copy_(p.grad.reshape(-1))
            off += n
        dist.all_reduce(self._flat, op=dist.ReduceOp.SUM, group=group)
        off = 0
        for p in self.params:
            n = p.numel()
            if p.grad is None:
                p.grad = self._flat[off:off + n].reshape(p.shape).clone()
            else:
                p.grad.copy_(self._flat[off:off + n].reshape(p.shape))
            off += n


def reduce_predictive_moments(sum_y: torch.Tensor, sum_y2: torch.Tensor, n_local: int, group=None):
    """Evaluation sharded by MC sample: combine per-rank sum_s y and sum_s y^2 into the
    predictive mean and (biased) variance over all samples."""
    count = torch.tensor([float(n_local)], device=sum_y.device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for t in (sum_y, sum_y2, count):
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    mean = sum_y / count
    var = sum_y2 / count - mean * mean
    return mean, var


def reduce_predictive_probs(prob_sum: torch.Tensor, loglik_sum: torch.Tensor | None, n_local: int, group=None):
    """Classification evaluation sharded by MC sample: combine per-rank sum_s softmax(z_s) (B, K) and sum_s log p_s(y) (B,)
    (``WHVIClassification.predictive_prob_sums``; ``loglik_sum`` may be None) into the MC-mean probabilities and the mean
    log-likelihood per input over all samples.  The test MNLL with n = m is minus the mean of the latter."""
    count = torch.tensor([float(n_local)], device=prob_sum.device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for t in (prob_sum, loglik_sum, count):
            if t is not None:
                dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return prob_sum / count, None if loglik_sum is None else loglik_sum / count


def reduce_predictive_uncertainty(prob_sum: torch.Tensor, ent_sum: torch.Tensor, logpred: torch.Tensor | None,
                                  loglik_sum: torch.Tensor | None, n_local: int, group=None):
    """Classification uncertainty with evaluation sharded by MC sample: combine each rank's sums of
    ``functional.categorical_uncertainty_`` (``WHVIClassification.predictive_uncertainty_sums``) over all samples.  prob_sum,
    ent_sum and loglik_sum are added across ranks (in place); logpred = log sum_s p_s(y) is combined as a log-sum-exp across
    ranks in fp64 (an all-reduce MAX, then a SUM of exp(l - max)): a row that is -inf on every rank stays -inf, and a NaN row on
    any rank (a label outside [0, K)) stays NaN.  Returns (``uncertainty.CategoricalUncertainty`` over all samples, the mean
    log-likelihood per input or None); logpred and loglik_sum may be None together.  Works in a single process too."""
    from .uncertainty import categorical_uncertainty
    count = torch.tensor([float(n_local)], dtype=torch.float64, device=prob_sum.device)
    logpred = None if logpred is None else logpred.to(torch.float64)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        for t in (prob_sum, ent_sum, loglik_sum, count):
            if t is not None:
                dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        if logpred is not None:
            nan = torch.isnan(logpred)
            finite = torch.where(nan, float("-inf"), logpred)
            m = finite.clone()
            dist.all_reduce(m, op=dist.ReduceOp.MAX, group=group)
            shift = torch.where(m == float("-inf"), 0.0, m)   # -inf everywhere: exp(-inf - 0) = 0, no -inf - -inf
            e = torch.exp(finite - shift)
            dist.all_reduce(e, op=dist.ReduceOp.SUM, group=group)
            any_nan = nan.to(torch.float64)
            dist.all_reduce(any_nan, op=dist.ReduceOp.SUM, group=group)
            logpred = torch.where(any_nan > 0, float("nan"), torch.log(e) + shift)
    S = int(count.item())
    return categorical_uncertainty(prob_sum, ent_sum, logpred, S), None if loglik_sum is None else loglik_sum / count.to(loglik_sum.dtype)
