"""WHVI weight parameterisations behind the reference's class names and signatures
(reference ``src/weights.py``): ``WHVISquarePow2Matrix``, ``WHVIStackedMatrix``,
``WHVIColumnMatrix``.  Parameter names, shapes, initialisation and registration order are
the reference's (``src/weights.py:28-32``), so ``state_dict`` KEYS AND SHAPES are interchangeable.
The FUNCTION those parameters define is not, under the default ``semantics="paper"``: weights
trained by the reference were trained for the map the reference actually executes
(``D.diag(s1 g s2)``, SURVEY F1) and must be loaded into modules built with
``semantics="reference"`` to reproduce the reference's predictions and loss;
``load_state_dict`` on a ``"paper"`` module says so once (``WARN_ON_LOAD``).

What changed underneath: the reference materialises a D x D matrix per MC sample through
four FWHTs of D x D matrices and multiplies by it (``src/weights.py:73``, ``:93``); here a
whole batch of MC samples goes through ONE fused kernel launch per layer
(``functional.whvi_layer``), O(S.B.D log D) work and O(S.B.D) memory.

MC samples are a leading tensor axis instead of a Python loop: a layer called with a 2-D
``(B, n_in)`` input and ``mc_samples = S`` (set by ``WHVINetwork``) returns ``(S, B, n_out)``;
called with ``(S, B, n_in)`` it maps sample to sample.  Called standalone on a 2-D input
(``mc_samples`` unset) it behaves exactly like the reference: one draw, 2-D output.

``semantics``:
  * ``"paper"`` (default) -- W = S1 H diag(g) H S2, the docstring formula at
    ``src/weights.py:77`` and the north-star definition of the hot path.  NOT numerically
    compatible with reference-trained weights (a different function of the same parameters).
  * ``"reference"`` -- the op chain as the reference actually executes it
    (``src/weights.py:73``: both FWHTs act on rows, so W collapses to D.diag(s1 g s2),
    SURVEY F1), run literally with this repo's FWHT kernel in place of ``fwht_cuda``; for
    seed-for-seed comparisons with the reference.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as WF
from .fwht import FWHTFunction

_SEMANTICS = ("paper", "reference")

# load_state_dict into a semantics="paper" block warns once per process that reference-trained weights
# need semantics="reference"; set to False to silence it (e.g. when resuming this package's own checkpoints).
WARN_ON_LOAD = True
_warned_on_load = False


def _warn_paper_load(module, *args):
    global _warned_on_load
    if WARN_ON_LOAD and not _warned_on_load and module.semantics == "paper":
        _warned_on_load = True
        import warnings
        warnings.warn('whvi_b200: loading a state_dict into WHVI blocks built with semantics="paper" (W = S1 H diag(g) H S2). '
                      'Checkpoints trained by the reference implementation were trained for the map it actually executes '
                      '(D.diag(s1 g s2), SURVEY F1): construct the model with semantics="reference" to reproduce their '
                      'predictions and loss.  (whvi_b200.weights.WARN_ON_LOAD = False silences this.)', stacklevel=3)


def _next_pow2(n: int) -> int:
    return 1 << max(0, (int(n) - 1).bit_length())


def _rowscale(d: torch.Tensor, A: torch.Tensor) -> torch.Tensor:
    """diag(d) @ A (the reference's matmul_diag_left, src/utils.py:4-12)."""
    return d.unsqueeze(-1) * A


class WHVISquarePow2Matrix(nn.Module):
    def __init__(self, D, lambda_=1e-5, bias=False, *, semantics="paper", kl_mode=0, covariance="diag"):
        """Square WHVI matrix of size (D, D), D a power of two.

        :param int D: rows/columns; power of two.
        :param float lambda_: prior variance.
        :param boolean bias: add a (non-variational) bias after the linear map.
        :param str semantics: "paper" or "reference" (module docstring).
        :param int kl_mode: 0 = the reference's KL formula (sigma used as a variance,
            src/utils.py:49-71), 1 = the statistically consistent sigma^2 form.
        :param str covariance: "diag" -- the reference's posterior, g = mu + softplus(rho) * eps (src/weights.py:43-50);
            "dense" -- superset: g = mu + L eps with a lower-triangular ``g_L`` (D, D) parameter in place of ``g_rho``
            (PAPER semantics), reparameterisation / its backward / the KL with log-determinant on the kernels of
            ``csrc/reparam_dense.cu`` (tcgen05 GEMMs at D >= 128, CUDA cores below).  Not in the reference: state_dicts
            differ (``g_L``).
        """
        super().__init__()
        if D < 1 or D & (D - 1):
            raise ValueError(f"D must be a power of two, got {D}")
        if semantics not in _SEMANTICS:
            raise ValueError(f"semantics must be one of {_SEMANTICS}")
        self.D = D
        self.lambda_ = lambda_
        self.padding = 0
        if covariance not in ("diag", "dense"):
            raise ValueError('covariance must be "diag" or "dense"')
        if covariance == "dense" and semantics != "paper":
            raise ValueError('covariance="dense" needs semantics="paper"')
        self.semantics = semantics
        self.kl_mode = kl_mode
        self.covariance = covariance
        self.mc_samples = None      # set by WHVINetwork while it runs a forward pass
        self._eps_queue = []        # injected noise, consumed first-in first-out

        # same registration and RNG draw order as src/weights.py:28-32
        self.bias = nn.Parameter(torch.zeros(1, D)) if bias else None
        self.s1 = nn.Parameter(torch.randn(D) * 0.01)
        self.s2 = nn.Parameter(torch.randn(D) * 0.01)
        self.g_mu = nn.Parameter(torch.zeros(D))
        g_rho = torch.rand(D) - 3
        if covariance == "dense":   # start from the reference's diagonal posterior: L = diag(softplus(rho))
            self.g_L = nn.Parameter(torch.diag(F.softplus(g_rho)))
        else:
            self.g_rho = nn.Parameter(g_rho)
        self._register_load_state_dict_pre_hook(_warn_paper_load, with_module=True)

    # ------------------------------------------------------------------ noise
    def inject_eps(self, eps: torch.Tensor) -> None:
        """Queue an ``(S, D)`` (or ``(D,)``) noise tensor for the next forward call."""
        self._eps_queue.append(eps.reshape(-1, self.D))

    def _draw_eps(self, S: int) -> torch.Tensor:
        if self._eps_queue:
            eps = self._eps_queue.pop(0).to(device=self.g_mu.device, dtype=torch.float32)
            if eps.size(0) != S:
                raise RuntimeError(f"injected eps has {eps.size(0)} samples, the forward pass needs {S}")
            return eps
        return torch.randn(S, self.D, device=self.g_mu.device)

    # ------------------------------------------------------------------ reference surface
    def fwht(self, x):
        return FWHTFunction.apply(x)

    @property
    def g_sigma(self):
        """Standard deviations of g: softplus(g_rho) (src/weights.py:43-50); dense: the diagonal of L."""
        return torch.diagonal(self.g_L) if self.covariance == "dense" else F.softplus(self.g_rho)

    def _g(self, eps):
        """(S, D) reparameterised samples of g for noise eps (S, D)."""
        if self.covariance == "dense":
            return WF.reparam_dense(self.g_mu, self.g_L, eps)
        return WF.reparam(self.g_mu, self.g_rho, eps)

    @property
    def kl(self):
        """KL from the N(0, lambda I) prior to the posterior of g (src/weights.py:52-64)."""
        if self.g_mu.device.type != "cuda":
            raise RuntimeError("whvi_b200 runs on CUDA only (no CPU fallback); move the module to a GPU")
        if self.covariance == "dense":
            return WF.kl_gaussian_dense(self.g_mu, self.g_L, self.lambda_)
        return WF.kl_gaussian(self.g_mu, self.g_rho, self.lambda_, self.kl_mode)

    def w_bar(self, u):
        """Dense D x D matrix S1 H diag(u) H S2 ("paper") or the as-written chain."""
        if self.semantics == "reference":
            return _rowscale(self.s1, self.fwht(_rowscale(u, self.fwht(torch.diag(self.s2)))))
        eye = torch.eye(self.D, device=u.device)
        return WF.whvi_layer(eye, u.reshape(1, self.D), self.s1, self.s2)[0].t()

    def sample(self):
        """One dense sample W (D x D)."""
        eps = self._draw_eps(1)
        if self.covariance == "dense":
            return self.w_bar(self._g(eps)[0])
        return self.w_bar(self.g_mu + self.g_sigma * eps[0])

    def _resolve_samples(self, x):
        if x.dim() == 3:
            return x.size(0), False
        if x.dim() != 2:
            raise RuntimeError("input must be (batch, D) or (samples, batch, D)")
        if self.mc_samples is None:
            return 1, True
        return int(self.mc_samples), False

    def sample_lrt(self, h, *, bias=None, relu_out=False, relu_in=False, dy_scale_from=None):
        """W h for a fresh draw of g per MC sample (local reparameterisation).  The
        keyword arguments are the kernel-side fusions (bias add, ReLU on the way out, ReLU
        mask on the way back); they default to the reference's plain behaviour.  A bfloat16 ``h`` gives a bfloat16
        result (bf16 activations, fp32 parameters and arithmetic; PAPER semantics only)."""
        if h.dtype == torch.bfloat16 and self.semantics == "reference":
            raise RuntimeError('WHVISquarePow2Matrix: bf16 activations are not supported with semantics="reference"')
        S, squeeze = self._resolve_samples(h)
        eps = self._draw_eps(S)
        if self.semantics == "reference":
            y = self._as_written(h, eps)
            if bias is not None:
                y = y + bias
            if relu_out:
                y = F.relu(y)
        else:
            g = self._g(eps)
            y = WF.whvi_layer(h, g, self.s1, self.s2, None if bias is None else bias.reshape(-1), relu_out, relu_in,
                              dy_scale_from)
        return y[0] if squeeze else y

    @property
    def fusable(self):
        """True when the fused-neighbour paths (ReLU / MNLL folded into the kernels) apply."""
        return self.semantics == "paper" and WF.MIN_LAYER_D <= self.D <= WF.FUSED_BWD_MAX_D  # the fused backward's range

    def forward_sqerr(self, h, target, *, relu_in=False):
        """Forward pass fused with sum (y - target)^2 (see functional.WHVILayerSqErrFunction).
        h: (B, D) or (S, B, D); target: (B, D).  Returns ((S, B, D) predictions, 0-d sum).
        bf16 ``h``: the bf16 forward, and the sum in torch from the widened predictions (the fused kernel is fp32 only)."""
        if h.dtype == torch.bfloat16:
            y = self.sample_lrt(h, bias=self.bias, relu_in=relu_in)
            return y, (y.float() - target).square().sum()
        S, _ = self._resolve_samples(h)
        g = self._g(self._draw_eps(S))
        bias = None if self.bias is None else self.bias.reshape(-1)
        return WF.whvi_layer_sqerr(h, g, self.s1, self.s2, bias, target, relu_in)

    def forward_loss(self, h, target, *, relu_in=False, dx_scale_to=None):
        """Training-time fused last layer: sum (y - target)^2 with the layer's backward computed in
        the same pass (functional.WHVILayerLossFunction).  Returns the 0-d sum only."""
        S, _ = self._resolve_samples(h)
        g = self._g(self._draw_eps(S))
        bias = None if self.bias is None else self.bias.reshape(-1)
        return WF.whvi_layer_loss(h, g, self.s1, self.s2, bias, target, relu_in, dx_scale_to)

    def predictive_moments(self, x, n_samples=64, *, chunk_samples=16, sample_range=None, out=None, generator=None, t2=None,
                           scatter_to=None):
        """MC predictive sums (sum_s y, sum_s y^2, samples done) for inputs x (B, D) without the
        (S, B, D) tensor: see functional.predictive_moments (BASELINE config 5, SURVEY 8f N1)."""
        if self.semantics != "paper":
            raise RuntimeError("predictive_moments implements the PAPER formula")
        eps = self._eps_queue.pop(0).to(device=self.g_mu.device, dtype=torch.float32) if self._eps_queue else None
        bias = None if self.bias is None else self.bias.reshape(-1)
        dense = self.covariance == "dense"
        return WF.predictive_moments(x, self.g_mu, None if dense else self.g_rho, self.s1, self.s2, bias, n_samples=n_samples,
                                     chunk_samples=chunk_samples, eps=eps, sample_range=sample_range, out=out,
                                     generator=generator, t2=t2, scatter_to=scatter_to, L=self.g_L if dense else None)

    @property
    def loss_fusable(self):
        return self.fusable and WF.LOSS_LAYER_MIN_D <= self.D <= WF.LOSS_LAYER_MAX_D

    def _as_written(self, h, eps):
        """src/weights.py:93 per sample: h @ (w_bar(mu) + w_bar(sigma*eps)).T"""
        outs = []
        w_mu = self.w_bar(self.g_mu)
        for s in range(eps.size(0)):
            W = w_mu + self.w_bar(self.g_sigma * eps[s])
            hs = h if h.dim() == 2 else h[s]
            outs.append(hs @ W.T)
        return torch.stack(outs)

    def forward(self, x, use_lrt=True, *, relu_out=False, relu_in=False, dy_scale_from=None):
        """x: (batch, D) or (samples, batch, D).  ``use_lrt`` is kept for signature
        compatibility; both branches of the reference compute W x for a sampled W."""
        return self.sample_lrt(x, bias=self.bias, relu_out=relu_out, relu_in=relu_in, dy_scale_from=dy_scale_from)


class WHVIStackedMatrix(nn.Module):
    def __init__(self, n_in, n_out, lambda_=1e-5, bias=False, *, semantics="paper", kl_mode=0, covariance="diag"):
        """Non-square WHVI matrix as a stack of square blocks (src/weights.py:111-133).  ``covariance`` as for
        ``WHVISquarePow2Matrix``, applied to every block: "dense" gives each block its own ``g_L``."""
        super().__init__()
        self.n_in = n_in
        self.n_out = n_out
        self.lambda_ = lambda_
        self.D_in, self.D_out, self.padding, self.stack = self.setup_dimensions(n_in, n_out)
        self.weight_matrices = nn.ModuleList([
            WHVISquarePow2Matrix(self.D_in, lambda_=lambda_, semantics=semantics, kl_mode=kl_mode, covariance=covariance)
            for _ in range(self.stack)
        ])
        self.bias = nn.Parameter(torch.zeros(1, self.D_out)) if bias else None
        self.one_launch = True   # False: block after block, as the reference does (tests compare the two)

    @staticmethod
    def setup_dimensions(D_in, D_out):
        """(D_in_adjusted, D_out_adjusted, padding, stack) as src/weights.py:135-160, with
        integer arithmetic (the reference's float log needs a fix-up branch, :151)."""
        D_adj = _next_pow2(D_in)
        padding = D_adj - D_in
        stack = -(-D_out // D_adj)
        return D_adj, D_adj * stack, padding, stack

    @property
    def mc_samples(self):
        return self.weight_matrices[0].mc_samples

    @mc_samples.setter
    def mc_samples(self, value):
        for w in self.weight_matrices:
            w.mc_samples = value

    # ------------------------------------------------------------------ one-launch path
    @property
    def grouped(self):
        """True when all blocks run as ONE grouped call per direction (functional.WHVIStackedFunction; with the dense posterior
        the grouped dense reparameterisation and functional.WHVIStackedGFunction): PAPER semantics, block size inside the fused
        kernels' range.  Otherwise block after block, as the reference does."""
        w = self.weight_matrices[0]
        return self.one_launch and w.semantics == "paper" and w.fusable

    fusable = grouped   # WHVINetwork folds a following nn.ReLU into the grouped launch
    loss_fusable = False

    def _pack(self):
        """Re-home the blocks' parameters into one (G, 4, D) buffer so that the kernels read them where they lie (evenly
        spaced); a no-op when they already are (after the first call, or once FlatParams owns them).  Same values, same
        Parameter objects, same state_dict -- only ``.data`` moves, like FlatParams does.  Dense blocks: s1, s2, g_mu and
        g_L of block k lie together, each segment on a 16-byte boundary (FlatParams' layout of one block)."""
        ws = self.weight_matrices
        if ws[0].covariance == "dense":
            vec_strides = {WF.uniform_stride([getattr(w, n) for w in ws]) for n in ("s1", "s2", "g_mu")}
            if None not in vec_strides and len(vec_strides) == 1 and WF.uniform_stride([w.g_L for w in ws]) is not None:
                return
            D = self.D_in
            v4, l4 = (D + 3) // 4 * 4, (D * D + 3) // 4 * 4
            with torch.no_grad():
                store = torch.empty((len(ws), 3 * v4 + l4), dtype=torch.float32, device=ws[0].s1.device)
                for k, w in enumerate(ws):
                    for i, n in enumerate(("s1", "s2", "g_mu", "g_L")):
                        p = getattr(w, n)
                        dst = store[k, i * v4:i * v4 + p.numel()].view(p.shape)
                        dst.copy_(p)
                        p.data = dst
            return
        names = ("s1", "s2", "g_mu", "g_rho")
        strides = [WF.uniform_stride([getattr(w, n) for w in ws]) for n in names]
        if None not in strides and len(set(strides)) == 1:
            return
        with torch.no_grad():
            store = torch.empty((len(ws), 4, self.D_in), dtype=torch.float32, device=ws[0].s1.device)
            for k, w in enumerate(ws):
                for i, n in enumerate(names):
                    p = getattr(w, n)
                    store[k, i].copy_(p)
                    p.data = store[k, i]

    def _eps_blocks(self, S):
        ws = self.weight_matrices
        if any(w._eps_queue for w in ws):   # injected noise (reference draw order, tests): per block
            return torch.stack([w._draw_eps(S) for w in ws])
        return torch.randn(len(ws), S, self.D_in, device=ws[0].g_mu.device)

    @property
    def kl(self):
        ws = self.weight_matrices
        if self.grouped and ws[0].g_mu.device.type == "cuda":
            if ws[0].covariance == "dense":
                return WF.kl_gaussian_dense_grouped([w.g_mu for w in ws], [w.g_L for w in ws], self.lambda_)
            return WF.kl_gaussian_grouped([w.g_mu for w in ws], [w.g_rho for w in ws], self.lambda_, ws[0].kl_mode)
        return sum(weight.kl for weight in ws)

    def sample(self):
        return torch.cat([weight.sample() for weight in self.weight_matrices])

    def sample_lrt(self, h):
        return torch.cat([weight.sample_lrt(h) for weight in self.weight_matrices], dim=-1)

    def forward(self, x, use_lrt=True, *, relu_out=False, relu_in=False):
        """x: (..., n_in) -> (..., n_out): zero-pad to D_in, apply every block, concatenate,
        add the bias, drop the padding outputs (src/weights.py:182-208).  A bfloat16 ``x`` gives a bfloat16 result (bf16
        activations, fp32 parameters and arithmetic) on the grouped path."""
        if x.dtype == torch.bfloat16:
            if x.device.type != "cuda":
                raise RuntimeError("WHVIStackedMatrix: bf16 activations run on CUDA only; move the module and its inputs to a GPU")
            if not self.grouped:
                raise RuntimeError('WHVIStackedMatrix: bf16 activations need the grouped path (semantics="paper", '
                                   f"4 <= D_in <= {WF.FUSED_BWD_MAX_D}, one_launch)")
        if self.grouped:
            if x.device.type != "cuda":
                raise RuntimeError("whvi_b200 runs on CUDA only (no CPU fallback); move the module and its inputs to a GPU")
            ws = self.weight_matrices
            S, squeeze = ws[0]._resolve_samples(x)
            self._pack()
            if ws[0].covariance == "dense":
                g = WF.reparam_dense_grouped([w.g_mu for w in ws], [w.g_L for w in ws], self._eps_blocks(S))
                y = WF.whvi_stacked_g(x, g, self.bias, self.n_out, [w.s1 for w in ws], [w.s2 for w in ws], relu_out, relu_in)
            else:
                y = WF.whvi_stacked(x, self._eps_blocks(S), self.bias, self.n_out, [w.s1 for w in ws], [w.s2 for w in ws],
                                    [w.g_mu for w in ws], [w.g_rho for w in ws], relu_out, relu_in)
            return y[0] if squeeze else y
        x_padded = F.pad(x, (0, self.D_in - self.n_in)) if self.D_in != self.n_in else x
        output = self.sample_lrt(x_padded)
        if self.bias is not None:
            output = output + self.bias
        output = output[..., :self.n_out]
        return F.relu(output) if relu_out else output


class WHVIColumnMatrix(nn.Module):
    def __init__(self, n_out, lambda_=1e-5, bias=False, transposed=False, *, semantics="paper", kl_mode=0, covariance="diag"):
        """Single-column (or, transposed, single-row) WHVI matrix (src/weights.py:211-229).  ``covariance`` as for
        ``WHVISquarePow2Matrix``, applied to the square block."""
        super().__init__()
        self.D = n_out
        self.D_adjusted = _next_pow2(n_out)
        self.weight_submodule = WHVISquarePow2Matrix(self.D_adjusted, lambda_=lambda_, semantics=semantics,
                                                     kl_mode=kl_mode, covariance=covariance)
        self.transposed = transposed
        self.bias = nn.Parameter(torch.zeros(1, 1 if transposed else n_out)) if bias else None
        self.one_launch = True   # False: the op chain of round 1 (FWHT of g + torch products); tests compare the two
        self.loss_fusable = False

    @property
    def mc_samples(self):
        return self.weight_submodule.mc_samples

    @mc_samples.setter
    def mc_samples(self, value):
        self.weight_submodule.mc_samples = value

    @property
    def kl(self):
        return self.weight_submodule.kl

    def _weights(self, S):
        """(S, D): the first D entries of the flattened sampled matrix, i.e. of its row 0
        (src/weights.py:239-245).  "paper": W[0, j] = s1[0] * s2[j] * (H g)[j], one FWHT of
        g per sample instead of a D x D sample."""
        sub = self.weight_submodule
        eps = sub._draw_eps(S)
        if sub.semantics == "reference":
            rows = [sub.w_bar(sub.g_mu + sub.g_sigma * eps[s]).reshape(-1)[:self.D] for s in range(S)]
            return torch.stack(rows)
        return (sub.s1[0] * sub.s2 * FWHTFunction.apply(sub._g(eps)))[:, :self.D]

    def sample(self):
        w = self._weights(1)[0].reshape(-1, 1)
        return w.T if self.transposed else w

    @property
    def fused(self):
        """True when the layer runs as one C-ABI call per direction (functional.WHVIColumnFunction; with the dense posterior
        the dense reparameterisation and functional.WHVIColumnGFunction): PAPER semantics."""
        sub = self.weight_submodule
        return self.one_launch and sub.semantics == "paper"

    def forward(self, x, *, relu_out=False, relu_in=False):
        """A bfloat16 ``x`` runs the fused path with bf16 activations: the plain form (1 -> n) returns bfloat16, the transposed
        form (n -> 1) float32 -- its (S, B, 1) output holds the network's predictions, which are not rounded to bf16."""
        if x.dtype == torch.bfloat16:
            if x.device.type != "cuda":
                raise RuntimeError("WHVIColumnMatrix: bf16 activations run on CUDA only; move the module and its inputs to a GPU")
            if not self.fused:
                raise RuntimeError('WHVIColumnMatrix: bf16 activations need the fused path (semantics="paper", one_launch)')
        sub = self.weight_submodule
        S, squeeze = sub._resolve_samples(x)
        if self.fused:
            if x.device.type != "cuda":
                raise RuntimeError("whvi_b200 runs on CUDA only (no CPU fallback); move the module and its inputs to a GPU")
            if sub.covariance == "dense":
                y = WF.whvi_column_g(x, sub._g(sub._draw_eps(S)), sub.s1, sub.s2, self.bias, self.D, self.transposed, relu_out,
                                     relu_in)
            else:
                y = WF.whvi_column(x, sub._draw_eps(S), sub.g_mu, sub.g_rho, sub.s1, sub.s2, self.bias, self.D, self.transposed,
                                   relu_out, relu_in)
            return y[0] if squeeze else y
        if relu_in:
            raise RuntimeError("relu_in needs the fused Column path")
        w = self._weights(S)                                   # (S, D)
        if self.transposed:                                    # (.., D) -> (.., 1)
            if x.dim() == 2:
                y = (x @ w.t()).t().unsqueeze(-1)              # (S, B, 1)
            else:
                y = torch.bmm(x, w.unsqueeze(-1))              # (S, B, 1)
        else:                                                  # (.., 1) -> (.., D)
            xs = x.unsqueeze(0) if x.dim() == 2 else x         # (1|S, B, 1)
            y = xs * w.unsqueeze(1)                            # (S, B, D)
        if self.bias is not None:
            y = y + self.bias
        if relu_out:
            y = F.relu(y)
        return y[0] if squeeze else y
