"""``WHVINetwork`` / ``WHVIRegression`` with the reference's signatures
(``src/networks.py``): forward -> ``(batch, out, n_samples)``, ``loss`` (ELBO),
``train_model`` (two-phase loop), ``eval_model``.

The reference runs the whole ``nn.Sequential`` once per MC sample in a Python loop
(``src/networks.py:48``).  Here the MC samples are a leading tensor axis: the sequence runs
ONCE, every WHVI layer handles all S samples in one fused kernel launch, and foreign
modules (``nn.Linear``, activations, ...) see the samples folded into the batch.
"""
from __future__ import annotations

import pathlib
from typing import Iterable, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as WF
from .layers import WHVI, WHVIConv2d, WHVILinear
from .likelihoods import CategoricalLikelihood, GaussianLikelihood, Likelihood

try:  # progress bars exactly like the reference when tqdm is around
    from tqdm import tqdm
except Exception:  # pragma: no cover
    def tqdm(it, **kwargs):
        return it


class WHVINetwork(nn.Module, WHVI):
    def __init__(self, modules: Iterable[nn.Module], likelihood: Likelihood, train_samples=1, eval_samples=64, *,
                 rng_mode="batched", fuse=True):
        """
        :param modules: modules for the underlying ``nn.Sequential``.
        :param likelihood: likelihood used in training.
        :param int train_samples: MC samples per forward pass in training mode.
        :param int eval_samples: MC samples per forward pass in eval mode.
        :param str rng_mode: "batched" draws one ``randn(S, D)`` per weight block;
            "reference" draws ``randn(D)`` per (sample, layer, block) in the reference's loop
            order (``src/networks.py:48`` -> ``src/weights.py:180`` -> ``:92``) so that the same
            seed yields the same noise as the reference.
        :param bool fuse: fold ``nn.ReLU`` between square WHVI layers and the Gaussian MNLL
            after a final square WHVI layer into the layer kernels (same numbers, fewer HBM
            round trips).  ``False`` runs every module as its own op, like the reference.
        """
        super().__init__()
        if rng_mode not in ("batched", "reference"):
            raise ValueError("rng_mode must be 'batched' or 'reference'")
        self.sequential = nn.Sequential(*modules)
        self.likelihood = likelihood
        self.train_samples = train_samples
        self.eval_samples = eval_samples
        self.rng_mode = rng_mode
        self.fuse = fuse
        self.current_mnll = 0.0
        self.current_kl = 0.0

    @property
    def kl(self):
        return sum([m.kl for m in self.sequential.children() if 'kl' in dir(m)])

    def _whvi_layers(self):
        return [m for m in self.sequential.children() if isinstance(m, (WHVILinear, WHVIConv2d))]

    def _predraw_reference_order(self, n_samples: int) -> None:
        blocks = [b for layer in self._whvi_layers() for b in layer.square_blocks()]
        draws = [[] for _ in blocks]
        for _ in range(n_samples):
            for i, b in enumerate(blocks):
                draws[i].append(torch.randn(b.D, device=b.g_mu.device))
        for b, d in zip(blocks, draws):
            b.inject_eps(torch.stack(d))

    @staticmethod
    def _fusable_square(module):
        from .weights import WHVISquarePow2Matrix
        return (isinstance(module, WHVILinear) and isinstance(module.weight_submodule, WHVISquarePow2Matrix)
                and module.weight_submodule.fusable)

    @staticmethod
    def _fusable_stacked(module):
        from .weights import WHVIStackedMatrix
        return isinstance(module, WHVILinear) and isinstance(module.weight_submodule, WHVIStackedMatrix) and module.weight_submodule.grouped

    @staticmethod
    def _fusable_column(module):
        from .weights import WHVIColumnMatrix
        return isinstance(module, WHVILinear) and isinstance(module.weight_submodule, WHVIColumnMatrix) and module.weight_submodule.fused

    @classmethod
    def _relu_fusable(cls, module):
        """Layers whose kernels can apply the mask of a ReLU folded into their producer to their dx (consumer side)."""
        return (cls._fusable_square(module) or cls._fusable_stacked(module)
                or (cls._fusable_column(module) and module.weight_submodule.transposed))

    def _run(self, x: torch.Tensor, n_samples: int, sqerr_target=None):
        """Run the sequence once with the MC samples as a leading axis.  Returns the
        (S, B, out) activations, or -- with ``sqerr_target`` and a fusable last layer --
        ``(activations, sum of squared errors)`` with the reduction done in the last
        layer's kernel.  ``[Square WHVI layer, nn.ReLU, Square WHVI layer]`` runs are executed
        with the ReLU folded into the two kernels (``self.fuse``).  Foreign modules before the first WHVI layer see the
        input as it is (e.g. a (B, C, H, W) image batch); after it, the sample axis folded into the batch."""
        modules = list(self.sequential.children())
        layers = self._whvi_layers()
        if self.rng_mode == "reference":
            self._predraw_reference_order(n_samples)
        for layer in layers:
            layer.mc_samples = n_samples
        sq = None
        try:
            h, i, relu_in, scale_holder = x, 0, False, None
            sampled = False   # a WHVI layer has run: h carries the sample axis
            while i < len(modules):
                module = modules[i]
                last = i == len(modules) - 1
                whvi_layer = isinstance(module, (WHVILinear, WHVIConv2d))
                sampled = sampled or whvi_layer
                if self.fuse and self._fusable_stacked(module):
                    # all blocks of the Stacked layer in one grouped launch, the following ReLU folded in when the
                    # consumer's kernels can apply the mask on the way back
                    relu_out = (i + 2 < len(modules) and type(modules[i + 1]) is nn.ReLU and self._relu_fusable(modules[i + 2]))
                    h = module.weight_submodule.forward(h, relu_out=relu_out, relu_in=relu_in)
                    relu_in, scale_holder = relu_out, None
                    i += 2 if relu_out else 1
                    continue
                if self.fuse and self._fusable_column(module):
                    w = module.weight_submodule   # (.., n) -> (.., 1) consumes a folded ReLU; (.., 1) -> (.., n) can produce one
                    relu_out = (not w.transposed and i + 2 < len(modules) and type(modules[i + 1]) is nn.ReLU
                                and self._relu_fusable(modules[i + 2]))
                    h = w.forward(h, relu_out=relu_out, relu_in=relu_in)
                    relu_in, scale_holder = relu_out, None
                    i += 2 if relu_out else 1
                    continue
                if self.fuse and self._fusable_square(module):
                    w = module.weight_submodule
                    relu_out = (i + 2 < len(modules) and type(modules[i + 1]) is nn.ReLU
                                and self._relu_fusable(modules[i + 2]))
                    if last and sqerr_target is not None and w.loss_fusable and torch.is_grad_enabled():
                        # training: forward + residual + backward of the last layer in one pass; its dx is
                        # for a unit loss coefficient, which the producer of h applies (scale_holder)
                        sq = w.forward_loss(h, sqerr_target, relu_in=relu_in, dx_scale_to=scale_holder)
                        h = None
                    elif last and sqerr_target is not None:
                        h, sq = w.forward_sqerr(h, sqerr_target, relu_in=relu_in)
                    else:
                        # h's only consumer will be the fused loss layer: share a DeferredScale with it
                        nxt = modules[i + 2].weight_submodule if relu_out else None
                        scale_holder = (WF.DeferredScale() if (relu_out and i + 2 == len(modules) - 1 and sqerr_target is not None
                                                               and nxt.loss_fusable and torch.is_grad_enabled()) else None)
                        h = w.forward(h, relu_out=relu_out, relu_in=relu_in, dy_scale_from=scale_holder)
                    relu_in = relu_out
                    i += 2 if relu_out else 1
                    continue
                if whvi_layer or not sampled:
                    h = module(h)
                else:  # foreign module: fold the sample axis into the batch
                    S, B = h.shape[0], h.shape[1]
                    h = module(h.reshape(S * B, *h.shape[2:]))
                    h = h.reshape(S, B, *h.shape[1:])
                i += 1
        finally:
            for layer in layers:
                layer.mc_samples = None
        if h is not None and not sampled:  # no WHVI layer introduced a sample axis: S identical predictions
            h = h.unsqueeze(0).expand(n_samples, *h.shape)
        return (h, sq) if sqerr_target is not None else h

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """x: (batch_size, in_dim) or an image batch (batch_size, C, H, W) -> (batch_size, out_dim, n_samples)."""
        assert x.dim() in (2, 4), "Input shape must be (batch_size, in_dim) or (batch_size, C, H, W)"
        batch_size = x.size()[0]
        n_samples = self.train_samples if self.training else self.eval_samples
        h = self._run(x, n_samples)
        predictions = h.reshape(n_samples, batch_size, -1).permute(1, 2, 0)
        assert predictions.dim() == 3
        return predictions

    def loss(self, x: torch.Tensor, y: torch.Tensor, n: int, ignore_kl=False) -> torch.Tensor:
        """Negative ELBO: MNLL estimate + KL (``src/networks.py:56-69``).  With a Gaussian
        likelihood and a square WHVI layer at the end, the squared-error reduction and its
        gradient are fused into that layer's kernels."""
        modules = list(self.sequential.children())
        fused = (self.fuse and isinstance(self.likelihood, GaussianLikelihood) and modules
                 and self._fusable_square(modules[-1]) and x.dim() == 2 and y.dim() == 2
                 and y.size(1) == modules[-1].weight_submodule.D and y.size(0) == x.size(0) and y.is_cuda)
        if fused:
            n_samples = self.train_samples if self.training else self.eval_samples
            _, sq = self._run(x, n_samples, sqerr_target=y.contiguous().float())
            self.current_mnll = self.likelihood.mnll_from_sq_error(sq, m=y.size(0), n_out=y.size(1), n_mc=n_samples, n=n)
        elif isinstance(self.likelihood, CategoricalLikelihood):
            # the (S, B, K) logits as the last module leaves them: no (B, K, S) permute copy
            n_samples = self.train_samples if self.training else self.eval_samples
            self.current_mnll = self.likelihood.mnll_from_logits(y, self._run(x, n_samples), n)
        else:
            self.current_mnll = self.likelihood.mnll_batch_estimate(y, self(x), n)
        self.current_kl = self.kl
        return self.current_mnll + self.current_kl if not ignore_kl else self.current_mnll

    def train_model(self, data_loader, optimizer, scheduler, epochs1: int = 500, epochs2: int = 5000,
                    pbar_update_period=20, ignore_kl=False, checkpoint_dir=None, *, cuda_graph=False):
        """Two-phase training loop of the reference (``src/networks.py:71-99``).

        ``cuda_graph=True`` (SURVEY 8f N3) replays each step -- forward, ELBO, backward, optimizer
        -- as one captured CUDA graph per minibatch shape (``whvi_b200.graphs``); the optimizer
        must be capturable and the minibatches on the GPU.  The small models the reference trains
        are launch-bound, so this is where their time goes."""
        self.train()
        graphed = None
        if cuda_graph:
            from .graphs import GraphedStepCache
            graphed = GraphedStepCache(self, optimizer, n=len(data_loader.dataset), ignore_kl=ignore_kl, scheduled=True)
        self.likelihood.requires_grad = False
        for phase, epochs, label in ((1, epochs1, 'Fixed LH'), (2, epochs2, 'Optimized LH')):
            if phase == 2:
                self.likelihood.requires_grad = True
            pbar = tqdm(range(epochs), desc=f'[{label}] KL = {float(self.current_kl):.2f}, '
                                            f'MNLL = {float(self.current_mnll):.2f}')
            for epoch in pbar:
                for data_x, data_y in data_loader:
                    if graphed is not None:
                        graphed(data_x, data_y)
                        scheduler.step()
                        continue
                    loss = self.loss(data_x, data_y, n=len(data_loader.dataset), ignore_kl=ignore_kl)
                    loss.backward()
                    optimizer.step()
                    scheduler.step()
                    self.zero_grad(set_to_none=(phase == 1))
                if phase == 2 and epoch % 5000 == 0 and checkpoint_dir is not None:
                    torch.save(self.state_dict(), pathlib.Path(checkpoint_dir) / f'epoch-{epoch}.pth')
                if epoch % pbar_update_period == 0 and hasattr(pbar, "set_description"):
                    pbar.set_description(f'[{label}] KL = {float(self.current_kl):.2f}, '
                                         f'MNLL = {float(self.current_mnll):.2f}')
        self.eval()

    @torch.no_grad()
    def predictive_sums(self, X: torch.Tensor, n_samples: int | None = None):
        """(sum_s y_hat, sum_s y_hat^2, S) over the MC samples for inputs X, each (batch, out) -- the two reductions
        ``eval_model`` needs (MC mean for the RMSE, ``src/networks.py:131-132``; squared errors for the MNLL,
        ``src/likelihoods.py:18-29``) WITHOUT the (batch, out, S) prediction tensor when the network ends in a square
        WHVI layer: that layer runs with the reduction fused in (``functional.layer_moments_raw`` /
        ``predictive_moments``; SURVEY 8f N1, BASELINE config 5).  Returns None when the last layer is not one."""
        modules = list(self.sequential.children())
        if not (self.fuse and modules and self._fusable_square(modules[-1]) and X.dim() == 2 and X.is_cuda):
            return None
        S = int(n_samples if n_samples is not None else (self.train_samples if self.training else self.eval_samples))
        last = modules[-1].weight_submodule
        head = WHVINetwork.__new__(WHVINetwork)          # the modules before the last layer, same settings
        nn.Module.__init__(head)
        head.sequential, head.rng_mode, head.fuse = nn.Sequential(*modules[:-1]), self.rng_mode, self.fuse
        if self.rng_mode == "reference":
            raise RuntimeError("predictive_sums draws batched noise; use forward() with rng_mode='reference'")
        h = head._run(X, S) if len(modules) > 1 else X
        if h.dim() == 2 or (h.dim() == 3 and h.stride(0) == 0):   # no WHVI layer before: one input block for all samples
            hh = h if h.dim() == 2 else h[0]
            sum_y, sum_y2, _ = last.predictive_moments(hh.float().contiguous(), S)
            return sum_y, sum_y2, S
        h = h.float()   # bf16 activations: the head ran in bf16; the moments kernel is fp32 (the widening is exact)
        bias = None if last.bias is None else last.bias.reshape(-1)
        g = last._g(last._draw_eps(S))
        sum_y = torch.empty(h.shape[1:], dtype=torch.float32, device=h.device)
        sum_y2 = torch.empty_like(sum_y)
        if WF.FUSED_MOMENTS_MIN_D <= last.D <= WF.FUSED_MOMENTS_MAX_D:
            WF.layer_moments_raw(h, g, last.s1, last.s2, bias, sum_y, sum_y2)
        else:
            WF.mc_moments_(WF.layer_forward_raw(h, g, last.s1, last.s2, bias), sum_y, sum_y2, accumulate=False)
        return sum_y, sum_y2, S

    def eval_model(self, X_test: torch.Tensor, y_test: torch.Tensor, loss) -> Tuple[float, float]:
        """Test error (``loss(y_pred, y_true)``) and MNLL on test data."""
        self.eval()
        y_pred = self(X_test)
        test_mnll = self.likelihood.mnll_batch_estimate(y_test, y_pred, n=y_test.size()[0])
        test_error = loss(y_pred, y_test)
        return float(test_error), float(test_mnll)


def _rmse_of_mc_mean(y_pred, y_true):
    return torch.sqrt(F.mse_loss(y_pred.mean(dim=2).flatten(), y_true.flatten()))


class WHVIRegression(WHVINetwork):
    def __init__(self, modules: Iterable[nn.Module], sigma: float = 1.0, **kwargs):
        """WHVI network for regression with a Gaussian likelihood (``src/networks.py:118-128``)."""
        super().__init__(modules, likelihood=GaussianLikelihood(sigma), **kwargs)

    def eval_model(self, X_test: torch.Tensor, y_test: torch.Tensor, loss=_rmse_of_mc_mean) -> Tuple[float, float]:
        """RMSE of the MC mean and test MNLL (``src/networks.py:101-115``, ``:130-133``).  With the default loss and a
        network that ends in a square WHVI layer, both come from ``predictive_sums`` -- sum_s y_hat and sum_s y_hat^2
        reduced inside the last layer's kernel -- so the (batch, out, S) tensor of the reference never exists
        (BASELINE config 5 is 1M x 32768 x 256 floats).  Any other loss function gets the full prediction tensor."""
        if loss is _rmse_of_mc_mean and y_test.dim() == 2:
            self.eval()
            sums = self.predictive_sums(X_test)
            if sums is not None and sums[0].shape == y_test.shape:
                sum_y, sum_y2, S = sums
                y = y_test.to(torch.float64)
                mean = sum_y.to(torch.float64) / S
                rmse = torch.sqrt(((mean - y) ** 2).mean())
                # sum_{b,i,s} (y - y_hat)^2 = S y^2 - 2 y sum_s y_hat + sum_s y_hat^2
                sq = (S * y * y - 2.0 * y * sum_y.to(torch.float64) + sum_y2.to(torch.float64)).sum()
                m, n_out = y_test.shape
                mnll = self.likelihood.mnll_from_sq_error(sq.to(torch.float32), m=m, n_out=n_out, n_mc=S, n=m)
                return float(rmse), float(mnll)
        return super().eval_model(X_test, y_test, loss)


class WHVIClassification(WHVINetwork):
    def __init__(self, modules: Iterable[nn.Module], **kwargs):
        """WHVI network for classification: the last module's K outputs are the logits of a softmax likelihood
        (``CategoricalLikelihood``); targets are (batch,) int64 class labels on the GPU."""
        super().__init__(modules, likelihood=CategoricalLikelihood(), **kwargs)

    @torch.no_grad()
    def predictive_prob_sums(self, X: torch.Tensor, y: torch.Tensor | None = None, n_samples: int | None = None,
                        chunk_samples: int | None = None):
        """(sum_s softmax(z_s) (batch, K) fp32, sum_s log softmax(z_s)[y] (batch,) fp32 or None without ``y``, S) over the MC
        samples.  The network runs ``chunk_samples`` samples at a time (default 16) and the ``whvi_categorical_predictive``
        kernel continues the sums chunk after chunk in sample order, so the (S, batch, K) logits never exist at once and the
        result does not depend on the chunking."""
        S = int(n_samples if n_samples is not None else (self.train_samples if self.training else self.eval_samples))
        chunk = max(1, int(chunk_samples if chunk_samples is not None else 16))
        prob_sum = loglik_sum = None
        for s0 in range(0, S, chunk):
            logits = self._run(X, min(chunk, S - s0))
            if prob_sum is None:
                prob_sum = torch.empty(logits.shape[1:], dtype=torch.float32, device=logits.device)
                loglik_sum = None if y is None else torch.empty(logits.shape[1], dtype=torch.float32, device=logits.device)
            WF.categorical_predictive_(logits, y, prob_sum, loglik_sum, accumulate=s0 > 0)
        if prob_sum is None:
            raise RuntimeError("predictive_prob_sums needs n_samples >= 1")
        return prob_sum, loglik_sum, S

    @torch.no_grad()
    def predict_proba(self, X: torch.Tensor, n_samples: int | None = None, chunk_samples: int | None = None) -> torch.Tensor:
        """MC-mean class probabilities (batch, K): 1/S sum_s softmax(z_s), ``chunk_samples`` samples at a time."""
        prob_sum, _, S = self.predictive_prob_sums(X, None, n_samples, chunk_samples)
        return prob_sum / S

    def eval_model(self, X_test: torch.Tensor, y_test: torch.Tensor, loss=None) -> Tuple[float, float]:
        """Error rate of the MC-mean prediction and test MNLL (the training estimator with n = m).  Both come from the
        chunked predictive sums; a user-supplied ``loss(y_pred, y_true)`` gets the (batch, K, S) logits of ``forward()``
        instead, as in ``WHVINetwork.eval_model``."""
        self.eval()
        if loss is not None:
            return super().eval_model(X_test, y_test, loss)
        prob_sum, loglik_sum, S = self.predictive_prob_sums(X_test, y_test)
        error = (prob_sum.argmax(dim=1) != y_test).to(torch.float64).mean()
        mnll = -loglik_sum.to(torch.float64).sum() / S   # n / (m S) * sum_{b,s} -log p with n = m
        return float(error), float(mnll)
