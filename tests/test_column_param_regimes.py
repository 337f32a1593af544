"""The Column layer and the parameter-side kernels against fp64 in every work-split regime they run in.

csrc/column.cu (the Column layer) and csrc/params.cu (diagonal reparameterisation and its backward, the diagonal KL, plain and
grouped, and the fused Adam step) cut their work with a few host-side rules: a capped element-wise grid that turns into a
grid-stride loop, 8 batch or sample slices per CTA, a grid.y cap, one CTA for a whole reduction.  This file restates those rules
from the source (CPU, with the cited lines checked), picks shapes that reach each regime and checks that every (kernel,
regime) cell has one, then runs the kernels at those shapes against fp64 restatements with every output and the workspace
filled with NaN first (GPU), so an element, slice or sample a kernel skips shows up as NaN or as a large error.

References.  Column: ``O.reparam``, ``O.column_weight_paper`` (batched through ``O.fwht``) and ``O.reparam_bwd`` with the
Column backward written out below (``_column_ref``), which a CPU test ties to torch fp64 autograd of the same forward.  KL: the
grouped KL is ``sum_k O.kl(mu_k, rho_k)``.  Adam: an fp64 restatement of ``torch.optim.Adam``'s step, and a 50-step trajectory
against ``torch.optim.Adam(foreach=False)``.

Tolerances are max|got - ref| / max|ref| (``rel_err``) unless a test says otherwise: forward outputs and the
reparameterisation 1e-5; gradients 1e-4 (DESIGN section 2), tighter where written below.
"""
from __future__ import annotations

import copy
import io
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import rel_err

SMS = 148
CSRC = Path(__file__).resolve().parent.parent / "whvi_b200" / "csrc"


# ------------------------------------------------------------------------------------------------- launch geometry, restated
def _cdiv(a, b):
    return -(-a // b)


def ew_grid(total):
    """column.cu:207-212 (ew_grid): ceil(total / 256) CTAs of 256 threads, at most 148 * 16; past that a grid-stride loop."""
    return max(1, min(_cdiv(total, 256), SMS * 16))


def dw_grid(S, n):
    """column.cu:264: column_dw_kernel runs (ceil(n / 32), min(S, 65535)) CTAs; a CTA loops over samples blockIdx.y + k gridDim.y."""
    return _cdiv(n, 32), min(S, 65535)


def dbias_ctas(transposed, n):
    """column.cu:282-286: the transposed form's dbias (one column) is one CTA; the plain form's is ceil(n / 32) CTAs."""
    return 1 if transposed else _cdiv(n, 32)


def param_parts(D):
    """column.cu:305: column_param_kernel writes ceil(D / 256) partial sums, which column_ds1_kernel folds in one thread."""
    return _cdiv(D, 256)


def reparam_grid(S, D):
    """params.cu:143-145: reparam_diag_kernel runs (ceil(D / 256), min(S, 4096)) CTAs and loops over samples past 4096."""
    return _cdiv(D, 256), max(1, min(S, 4096))


REPARAM_BWD_SLICES = 8   # params.cu:53: reparam_diag_bwd_kernel's 8 warps take samples ty, ty + 8, ... (grid.y = groups, :154)


def kl_threads(D, G=1):
    """params.cu:163-165: launch_kl's single CTA has the next power of two of D * G threads, from 32 up to 1024."""
    t = 32
    while t < D * G and t < 1024:
        t <<= 1
    return t


def adam_grid(n):
    """params.cu:243-244: ceil(n / 256) CTAs, at most 148 * 8; past that a grid-stride loop."""
    return min(_cdiv(n, 256), SMS * 8)


# each citation above, and the source text it rests on
CITED = [("column.cu", 210, "if (b > 148 * 16) b = 148 * 16;"),
         ("column.cu", 264, "S < 65535 ? S : 65535"),
         ("column.cu", 284, "column_dbias_kernel<float><<<1, 256"),
         ("column.cu", 286, "(cols + 31) / 32"),
         ("column.cu", 305, "nparts = static_cast<int>((D + 255) / 256)"),
         ("params.cu", 145, "S > 4096 ? 4096 : S"),
         ("params.cu", 53, "s += 8"),
         ("params.cu", 154, "static_cast<unsigned>(groups)"),
         ("params.cu", 165, "while (threads < total && threads < 1024) threads <<= 1;"),
         ("params.cu", 244, "if (blocks > 148 * 8) blocks = 148 * 8;")]


def _dim(n):
    return 1 << (n - 1).bit_length()


def _up4(v):
    return _cdiv(v, 4) * 4


def column_ws_floats(S, D, n):
    """column.cu:250-254: dhg (S, D) | dg (S, D) | dwp (S, n) | partial sums, each segment rounded up to 4 floats."""
    return 2 * _up4(S * D) + _up4(S * n) + _up4(param_parts(D))


# ------------------------------------------------------------------------------------------------- the shapes
# Column: (S, B, n, transposed, shared x, relu, same-sign dy).  relu: RELU_IN on the transposed form, RELU_OUT on the plain
# form; either way about half the inputs are exactly 0.
COLUMN_SHAPES = [
    (3, 5, 20, True, False, True, False),          # n < 32, S B % 8, B < 8
    (2, 7, 100, True, True, False, False),         # n % 32, shared x
    (3, 9, 200, True, False, False, False),        # B % 8, one partial sum at D = 256
    (4, 300, 600, True, False, True, False),       # dot_dx grid-stride loop with RELU_IN
    (2, 1 << 21, 3, True, False, False, True),     # dbias: one CTA over 4.2e6 rows of same-sign dy
    (65537, 3, 5, True, False, False, False),      # S > 65535: dw's grid.y loop; reparam's grid.y loop
    (2, 3, 16385, True, False, False, False),      # D = 32768: 128 partial sums, n = D / 2 + 1
    (3, 5, 20, False, False, True, False),         # plain: n < 32, B < 8, RELU_OUT
    (2, 11, 1000, False, True, True, False),       # plain: n >> 32, shared x, dbias over 32 CTAs
    (3, 400, 700, False, False, True, False),      # plain: outer grid-stride loop with RELU_OUT, dbias over 22 CTAs
    (65537, 2, 3, False, False, False, False),     # plain: S > 65535
    (2, 5, 16385, False, True, False, False),      # plain: 128 partial sums
]
# bf16 Column calls of more than 2^31 activation elements: (S, B, n, transposed)
INT64_SHAPES = [(2, 1_073_742, 1000, True), (2, 1_073_742, 1000, False)]
# whvi_reparam_f32 / whvi_reparam_bwd_f32: (S, D)
REPARAM_SHAPES = [(5000, 100), (3, 50), (13, 1000), (64, 256), (1, 4097)]
# grouped reparameterisation through a Stacked call: (S, B, D, G, param_stride)
STACKED_REPARAM_SHAPES = [(1500, 1, 16, 3, 20), (3, 2, 16, 3, 20), (13, 1, 64, 2, 68)]
# KL: (D, G, param_stride, mode, grad_scale, accumulate); G = 0: whvi_kl_f32, else whvi_kl_grouped_f32 (no accumulate)
KL_SHAPES = [(20, 0, 0, 0, 1.0, 0), (20, 0, 0, 1, 0.375, 1), (700, 0, 0, 1, 1.0, 0), (700, 0, 0, 0, 2.5, 1),
             (5000, 0, 0, 0, 0.375, 0), (5000, 0, 0, 1, 1.0, 1),
             (8, 3, 8, 0, 1.0, 0), (8, 3, 12, 1, 0.375, 0), (100, 5, 104, 0, 2.5, 0), (100, 5, 100, 1, 1.0, 0),
             (1024, 3, 1028, 1, 0.375, 0), (1024, 3, 1024, 0, 1.0, 0)]
# Adam: n; and per n every (lr on the device, beta1, grad_scale) and every t of ADAM_STEPS
ADAM_SIZES = [100, 1000, 606_285]
ADAM_ARGS = [(False, 0.9, 1.0), (True, 0.9, 0.375), (False, 0.0, 2.5)]
ADAM_STEPS = [1, 2, 10, 1000, 10 ** 6]


# ------------------------------------------------------------------------------------------------- regimes
def column_cells(S, B, n, transposed, shared, relu, positive):
    D, rows, total = _dim(n), S * B, S * B * n
    c = set()
    if transposed:
        ew = "column_dot_dx"
        if n < 32:
            c.add(("column_dot", "n < 32"))
        if n >= 32 and n % 32:
            c.add(("column_dot", "n >= 32, n % 32 != 0"))
        if rows % 8:
            c.add(("column_dot", "S B % 8 != 0"))
        if shared:
            c.add(("column_dot", "shared x"))
    else:
        ew = "column_outer"
        if n < 32:
            c.add(("column_outer_dx", "n < 32"))
        if n >= 1024:
            c.add(("column_outer_dx", "n >> 32"))
    c.add((ew, "grid-stride" if ew_grid(total) * 256 < total else "one pass"))
    if relu:
        c.add((ew, "relu with x == 0"))
    if B < 8:
        c.add(("column_dw", "B < 8"))
    elif B % 8:
        c.add(("column_dw", "B % 8 != 0"))
    if n % 32:
        c.add(("column_dw", "n % 32 != 0"))
    if shared:
        c.add(("column_dw", "shared x, transposed" if transposed else "shared x, plain"))
    if dw_grid(S, n)[1] < S:
        c.add(("column_dw", "S > 65535"))
    if transposed and dbias_ctas(True, n) == 1 and rows >= 256 * 64:
        c.add(("column_dbias", "one CTA, S B >> 256 rows"))
        if positive:
            c.add(("column_dbias", "one CTA, same-sign dy"))
    if not transposed and n % 32 and dbias_ctas(False, n) >= 2:
        c.add(("column_dbias", "plain, n % 32 != 0, several CTAs"))
    if param_parts(D) == 1:
        c.add(("column_param", "one part"))
    if param_parts(D) == 128 and n == D // 2 + 1:
        c.add(("column_param", "128 parts, n = D / 2 + 1"))
    c |= reparam_cells(S, D)
    c |= reparam_bwd_cells(S, D, 0, 1)
    return c


def reparam_cells(S, D, grouped=False):
    c = set()
    if reparam_grid(S, D)[1] < S:
        c.add(("reparam", "S > 4096"))
    if grouped:
        c.add(("reparam", "grouped, param_stride > D"))
    if D % 256:
        c.add(("reparam", "D % 256 != 0"))
    return c


def reparam_bwd_cells(S, D, accumulate, groups):
    c = {("reparam_bwd", f"accumulate {accumulate}")}
    if S < REPARAM_BWD_SLICES:
        c.add(("reparam_bwd", "S < 8"))
    elif S % REPARAM_BWD_SLICES:
        c.add(("reparam_bwd", "S % 8 != 0"))
    if D % 32:
        c.add(("reparam_bwd", "D % 32 != 0"))
    if groups > 1:
        c.add(("reparam_bwd", "groups > 1"))
    return c


def kl_cells(D, G, pstride, mode, grad_scale, accumulate):
    total = D * max(G, 1)
    c = {("kl", f"mode {mode}")}
    c.add(("kl", "D G <= 32" if total <= 32 else "32 < D G <= 1024" if total <= 1024 else "D G > 1024"))
    if kl_threads(D, max(G, 1)) < total:
        c.add(("kl", "threads loop"))
    if G and pstride > D:
        c.add(("kl", "grouped, param_stride > D"))
    if G:
        c.add(("kl", "grouped"))
    if grad_scale != 1.0:
        c.add(("kl", "grad_scale != 1"))
    if accumulate:
        c.add(("kl", "accumulate"))
    return c


def adam_cells(n, lr_dev, b1, grad_scale):
    c = {("adam", "lr on the device" if lr_dev else "host lr")}
    if n < 256:
        c.add(("adam", "n < 256"))
    if n % 256:
        c.add(("adam", "n % 256 != 0"))
    if adam_grid(n) * 256 < n:
        c.add(("adam", "grid-stride"))
    if grad_scale != 1.0:
        c.add(("adam", "grad_scale != 1"))
    if b1 == 0.0:
        c.add(("adam", "beta1 = 0"))
    return c


def covered_cells():
    cells = set()
    for case in COLUMN_SHAPES:
        cells |= column_cells(*case)
    for S, B, n, transposed in INT64_SHAPES:
        if S * B * n > 1 << 31:
            cells.add(("int64", "transposed" if transposed else "plain"))
    for S, D in REPARAM_SHAPES:
        cells |= reparam_cells(S, D)
        for acc in (0, 1):
            cells |= reparam_bwd_cells(S, D, acc, 1)
    for S, B, D, G, pstride in STACKED_REPARAM_SHAPES:
        cells |= reparam_cells(S * G, D, grouped=pstride > D)
        cells |= reparam_bwd_cells(S, D, 0, G)
    for shape in KL_SHAPES:
        cells |= kl_cells(*shape)
    for n in ADAM_SIZES:
        for lr_dev, b1, gs in ADAM_ARGS:
            cells |= adam_cells(n, lr_dev, b1, gs)
    return cells


REQUIRED = {
    ("column_dot", "n < 32"), ("column_dot", "n >= 32, n % 32 != 0"), ("column_dot", "S B % 8 != 0"), ("column_dot", "shared x"),
    ("column_outer", "one pass"), ("column_outer", "grid-stride"), ("column_outer", "relu with x == 0"),
    ("column_dot_dx", "one pass"), ("column_dot_dx", "grid-stride"), ("column_dot_dx", "relu with x == 0"),
    ("column_dw", "B < 8"), ("column_dw", "B % 8 != 0"), ("column_dw", "n % 32 != 0"), ("column_dw", "shared x, transposed"),
    ("column_dw", "shared x, plain"), ("column_dw", "S > 65535"),
    ("column_outer_dx", "n < 32"), ("column_outer_dx", "n >> 32"),
    ("column_dbias", "one CTA, S B >> 256 rows"), ("column_dbias", "one CTA, same-sign dy"),
    ("column_dbias", "plain, n % 32 != 0, several CTAs"),
    ("column_param", "one part"), ("column_param", "128 parts, n = D / 2 + 1"),
    ("int64", "transposed"), ("int64", "plain"),
    ("reparam", "S > 4096"), ("reparam", "grouped, param_stride > D"), ("reparam", "D % 256 != 0"),
    ("reparam_bwd", "S < 8"), ("reparam_bwd", "S % 8 != 0"), ("reparam_bwd", "D % 32 != 0"), ("reparam_bwd", "accumulate 0"),
    ("reparam_bwd", "accumulate 1"), ("reparam_bwd", "groups > 1"),
    ("kl", "D G <= 32"), ("kl", "32 < D G <= 1024"), ("kl", "D G > 1024"), ("kl", "threads loop"), ("kl", "grouped"),
    ("kl", "grouped, param_stride > D"), ("kl", "mode 0"), ("kl", "mode 1"), ("kl", "grad_scale != 1"), ("kl", "accumulate"),
    ("adam", "n < 256"), ("adam", "n % 256 != 0"), ("adam", "grid-stride"), ("adam", "host lr"), ("adam", "lr on the device"),
    ("adam", "grad_scale != 1"), ("adam", "beta1 = 0"),
}


# ------------------------------------------------------------------------------------------------- CPU
def test_cited_launch_geometry_is_the_source():
    """Each restated rule cites a line of csrc/; the line still says it."""
    for name, line, text in CITED:
        src = (CSRC / name).read_text().splitlines()
        assert text in src[line - 1], f"{name}:{line} no longer reads {text!r}: {src[line - 1]!r}"


def test_restated_workspace_matches_library_query():
    """The workspace layout (and with it the partial-sum count ceil(D / 256)) against whvi_column_bwd_workspace_bytes."""
    from ctypes import byref, c_size_t
    from whvi_b200 import _lib
    L = _lib.lib()
    ws = c_size_t(0)
    shapes = {(S, _dim(n), n) for S, _, n, *_ in COLUMN_SHAPES} | {(S, _dim(n), n) for S, _, n, _ in INT64_SHAPES}
    shapes |= {(S, 1 << k, n) for k in range(0, 16) for S in (1, 3, 65537) for n in {(1 << k) // 2 + 1, 1 << k}}
    for S, D, n in sorted(shapes):
        _lib.check(L.whvi_column_bwd_workspace_bytes(S, D, n, byref(ws)), "whvi_column_bwd_workspace_bytes")
        assert ws.value == 4 * column_ws_floats(S, D, n), (S, D, n)


def test_every_regime_cell_is_covered():
    missing = sorted(REQUIRED - covered_cells())
    assert not missing, f"regime cells without a shape: {missing}"
    for S, B, n, *_ in COLUMN_SHAPES:    # every Column shape is a legal call: D = next_pow2(n), n > D / 2
        assert n > _dim(n) // 2 or n == 1
    for S, B, D, G, pstride in STACKED_REPARAM_SHAPES:
        assert pstride >= D and pstride % 4 == 0


# ------------------------------------------------------------------------------------------------- the fp64 Column restatement
def _column_weights(g, s1, s2, n):
    """w (S, n) = s1[0] s2[:n] (H g_s)[:n] for every sample, through the batched oracle FWHT; hg = H g."""
    from oracle import oracle as O
    hg = O.fwht(np.asarray(g, dtype=np.float64))
    w = s1[0] * s2[None, :n] * hg[:, :n]
    assert np.array_equal(w[0], O.column_weight_paper(g[0], s1, s2, n))
    return hg, w


def _column_bwd_params(dwp, hg, s1, s2, rho, eps, n):
    """From dwp = dL/dw (S, n) to the parameter side: dhg = dwp s1[0] s2 on j < n (0 past n); dg = H dhg;
    ds2 = s1[0] sum_s dwp hg (0 past n); ds1[0] = sum_j s2 q with q = sum_s dwp hg (ds1[1:] = 0); dmu, drho by O.reparam_bwd."""
    from oracle import oracle as O
    S, D = hg.shape
    dhg = np.zeros((S, D))
    dhg[:, :n] = dwp * s1[0] * s2[None, :n]
    dg = O.fwht(dhg)
    q = (dwp * hg[:, :n]).sum(0)
    ds2 = np.zeros(D)
    ds2[:n] = s1[0] * q
    ds1 = np.zeros(D)
    ds1[0] = (s2[:n] * q).sum()
    dmu, drho = O.reparam_bwd(rho, eps, dg)
    ds1_scale = (np.abs(s2[:n]) * np.abs(dwp * hg[:, :n]).sum(0)).sum()   # sum of |terms| of ds1[0] = sum_j,s s2 dwp hg
    return dict(dhg=dhg, dg=dg, ds1=ds1, ds2=ds2, dmu=dmu, drho=drho, ds1_scale=ds1_scale)


def _column_ref(x, dy, mu, rho, eps, s1, s2, bias, n, transposed, relu):
    """fp64 Column layer, forward and backward.  x: (S, B, width) or shared (B, width); dy: (S, B, 1) transposed,
    (S, B, n) plain.  Returns every output the kernels write, dx per sample."""
    from oracle import oracle as O
    g = O.reparam(mu, rho, eps)
    hg, w = _column_weights(g, s1, s2, n)
    S = eps.shape[0]
    xb = np.broadcast_to(x, (S,) + x.shape[-2:])
    if transposed:
        y = np.einsum("sbj,sj->sb", xb, w)[..., None] + bias[0]
        dx = dy * w[:, None, :] * (xb > 0 if relu else 1.0)   # RELU_IN: x is a ReLU's output, mask x > 0
        dwp = np.einsum("sb,sbj->sj", dy[..., 0], xb)
        dbias = np.array([dy.sum()])
    else:
        y = xb * w[:, None, :] + bias[None, None, :]
        if relu:   # RELU_OUT: dy is the gradient of the pre-activation (the next layer's RELU_IN masks it)
            y = np.maximum(y, 0.0)
        dx = np.einsum("sbj,sj->sb", dy, w)[..., None]
        dwp = np.einsum("sb,sbj->sj", xb[..., 0], dy)
        dbias = dy.sum((0, 1))
    out = dict(g=g, hg=hg, y=y, dx=dx, dwp=dwp, dbias=dbias)
    out.update(_column_bwd_params(dwp, hg, s1, s2, rho, eps, n))
    return out


def _column_case(case, seed):
    S, B, n, transposed, shared, relu, positive = case
    rng = np.random.default_rng(seed)
    D, width = _dim(n), n if transposed else 1
    x = _randn(rng, *((B, width) if shared else (S, B, width)))
    if relu:
        x = np.maximum(x, 0.0)
    dy = _randn(rng, S, B, 1 if transposed else n)
    if positive:
        dy = np.abs(dy)
    mu, rho, s1, s2 = (_randn(rng, D) for _ in range(4))
    eps = _randn(rng, S, D)
    bias = _randn(rng, 1 if transposed else n)
    return x, dy, mu, rho, eps, s1, s2, bias


def _randn(rng, *shape):
    """fp32 draws widened to fp64: the reference sees exactly the kernel's inputs."""
    return rng.standard_normal(shape, dtype=np.float32).astype(np.float64)


@pytest.mark.parametrize("transposed,shared,relu", [(True, False, True), (True, True, False), (False, False, True),
                                                    (False, True, False)])
def test_column_restatement_is_torch_autograd(transposed, shared, relu):
    """The restated Column backward (dx, dmu, drho, ds1, ds2, dbias) against torch fp64 autograd of the same forward
    (y = x w + bias with w = s1[0] s2[:n] (H (mu + softplus(rho) eps))[:n]), at a small shape."""
    from oracle import oracle as O
    S, B, n = 3, 6, 13
    D = _dim(n)
    x, dy, mu, rho, eps, s1, s2, bias = _column_case((S, B, n, transposed, shared, relu, False), 11)
    x = x - 0.25 if relu else x                    # some negative pre-activations for the ReLU to cut
    ref = _column_ref(np.maximum(x, 0.0) if (relu and transposed) else x, dy, mu, rho, eps, s1, s2, bias, n, transposed, relu)
    T = lambda a: torch.tensor(a, dtype=torch.float64, requires_grad=True)
    xt, mut, rhot, s1t, s2t, bt = T(x), T(mu), T(rho), T(s1), T(s2), T(bias)
    H = torch.tensor(O.build_H(D))
    hg = (mut + torch.nn.functional.softplus(rhot) * torch.tensor(eps)) @ H
    w = s1t[0] * s2t[:n] * hg[:, :n]
    xin = torch.relu(xt) if (relu and transposed) else xt
    xin = xin.expand((S,) + xin.shape[-2:])
    if transposed:
        y = pre = (xin * w[:, None, :]).sum(-1, keepdim=True) + bt[0]
    else:   # RELU_OUT: dy is the gradient of the pre-activation
        pre = xin * w[:, None, :] + bt
        y = torch.relu(pre) if relu else pre
    assert rel_err(y.detach().numpy(), ref["y"]) < 1e-13
    (pre * torch.tensor(dy)).sum().backward()
    dx = ref["dx"].sum(0) if shared else ref["dx"]
    for name, got, want in (("dx", xt.grad, dx), ("dmu", mut.grad, ref["dmu"]), ("drho", rhot.grad, ref["drho"]),
                            ("ds1", s1t.grad, ref["ds1"]), ("ds2", s2t.grad, ref["ds2"]), ("dbias", bt.grad, ref["dbias"])):
        assert rel_err(got.numpy(), want) < 1e-12, name


# ------------------------------------------------------------------------------------------------- GPU helpers
def dev():
    return torch.device("cuda:0")


def t(a, dtype=torch.float32):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev()).to(dtype)


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), dtype=dtype, device=dev())


def _close(got, ref, what, tol):
    got = got.double().cpu().numpy() if isinstance(got, torch.Tensor) else got
    err = rel_err(got, ref)
    assert err <= tol, f"{what}: rel err {err:.3e} > {tol:g}"


def _stream():
    from whvi_b200 import functional as F
    return F._stream(dev())


def _run_column(x, dy, mu, rho, eps, s1, s2, bias, S, B, n, transposed, relu, bf16):
    """One raw forward and one raw backward call with every output and the workspace NaN-filled first.  x, dy: device tensors
    (bf16 where the call takes bf16).  Returns the outputs and the workspace segments dhg, dg, dwp."""
    from whvi_b200 import _lib
    L = _lib.lib()
    D = _dim(n)
    width = n if transposed else 1
    xs = 0 if x.dim() == 2 else B * width
    act = torch.bfloat16 if bf16 else torch.float32
    g, hg = _nan(S, D), _nan(S, D)
    y = _nan(S, B, 1) if transposed else _nan(S, B, n, dtype=act)
    sfx = "bf16" if bf16 else "f32"
    rc = getattr(L, f"whvi_column_fwd_{sfx}")(x.data_ptr(), xs, mu.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(),
                                             eps.data_ptr(), bias.data_ptr(), g.data_ptr(), hg.data_ptr(), y.data_ptr(), S, B, D, n,
                                             int(transposed), int(relu and not transposed), _stream())
    _lib.check(rc, f"whvi_column_fwd_{sfx}")
    ws = _nan(column_ws_floats(S, D, n))
    dx = _nan(S, B, width, dtype=act)
    dmu, drho, ds1, ds2 = (_nan(D) for _ in range(4))
    dbias = _nan(1 if transposed else n)
    rc = getattr(L, f"whvi_column_bwd_{sfx}")(x.data_ptr(), xs, dy.data_ptr(), hg.data_ptr(), rho.data_ptr(), s1.data_ptr(),
                                             s2.data_ptr(), eps.data_ptr(), dx.data_ptr(), dmu.data_ptr(), drho.data_ptr(),
                                             ds1.data_ptr(), ds2.data_ptr(), dbias.data_ptr(), ws.data_ptr(), 4 * ws.numel(), S, B, D,
                                             n, int(transposed), int(relu and transposed), _stream())
    _lib.check(rc, f"whvi_column_bwd_{sfx}")
    torch.cuda.synchronize()
    o = _up4(S * D)
    return dict(g=g, hg=hg, y=y, dx=dx, dmu=dmu, drho=drho, ds1=ds1, ds2=ds2, dbias=dbias, dhg=ws[:S * D].view(S, D),
                dg=ws[o:o + S * D].view(S, D), dwp=ws[2 * o:2 * o + S * n].view(S, n))


# ------------------------------------------------------------------------------------------------- Column vs fp64
# rel_err bounds met by every shape above with room to spare; the gradients' are DESIGN section 2's 1e-4 unless tighter here
# (largest seen on a B200: g 8e-8, hg 1.5e-7, y 1.1e-6, dx 6e-7, the gradients up to 1.6e-5).  ds1 has one nonzero entry, a
# sum over j and s whose terms cancel: its bound is 1e-5 of the sum of the terms' magnitudes (ds1_scale), not of its value.
COLUMN_TOL = dict(g=1e-5, hg=1e-5, y=1e-5, dx=1e-5, dwp=1e-4, dbias=1e-4, dhg=1e-4, dg=1e-4, ds2=1e-4, dmu=1e-4, drho=1e-4)
DS1_TOL = 1e-5


def _ds1_close(got, ref, what):
    err = abs(float(got[0]) - ref["ds1"][0])
    assert err <= DS1_TOL * ref["ds1_scale"], f"{what}: |err| {err:.3e} > {DS1_TOL:g} x {ref['ds1_scale']:.3e}"
    assert torch.count_nonzero(got[1:]) == 0, f"{what}: ds1[1:] not exactly 0"


def _case_id(case):
    S, B, n, tr, shared, relu, pos = case
    return f"S{S}-B{B}-n{n}-{'T' if tr else 'P'}{'-shared' if shared else ''}{'-relu' if relu else ''}{'-pos' if pos else ''}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", COLUMN_SHAPES, ids=_case_id)
def test_column_vs_fp64(case):
    S, B, n, transposed, shared, relu, positive = case
    D = _dim(n)
    x, dy, mu, rho, eps, s1, s2, bias = _column_case(case, S * 7 + B * 13 + n)
    got = _run_column(t(x), t(dy), t(mu), t(rho), t(eps), t(s1), t(s2), t(bias), S, B, n, transposed, relu, False)
    ref = _column_ref(x, dy, mu, rho, eps, s1, s2, bias, n, transposed, relu)
    for name, tol in COLUMN_TOL.items():
        _close(got[name], ref[name], f"{name} {_case_id(case)}", tol)
    _ds1_close(got["ds1"], ref, f"ds1 {_case_id(case)}")
    # the parameter side past n is exactly zero: only s1[0] and s2[:n] enter row 0 of W
    assert torch.count_nonzero(got["ds2"][n:]) == 0
    assert torch.count_nonzero(got["dhg"][:, n:]) == 0
    if relu and transposed:   # RELU_IN: x == 0 gives dx exactly 0
        assert torch.count_nonzero(got["dx"][t(np.broadcast_to(x, (S,) + x.shape[-2:])) == 0]) == 0
    if relu and not transposed:
        assert bool((got["y"] >= 0).all())


@pytest.mark.gpu
@pytest.mark.parametrize("case", COLUMN_SHAPES, ids=_case_id)
def test_column_bf16_is_fp32_on_widened_inputs(case):
    """At every Column shape above: the bf16 call equals the fp32 call on the widened inputs, bit for bit (activation outputs
    rounded once; g, H g, the transposed form's y and every parameter gradient identical)."""
    S, B, n, transposed, shared, relu, positive = case
    x, dy, mu, rho, eps, s1, s2, bias = _column_case(case, S * 7 + B * 13 + n)
    xb = t(x, torch.bfloat16)
    dyb = t(dy) if transposed else t(dy, torch.bfloat16)
    p = [t(v) for v in (mu, rho, eps, s1, s2, bias)]
    b16 = _run_column(xb, dyb, *p[:5], p[5], S, B, n, transposed, relu, True)
    b32 = _run_column(xb.float(), dyb.float(), *p[:5], p[5], S, B, n, transposed, relu, False)
    for name in b16:
        a, b = b16[name], b32[name]
        if a.dtype == torch.bfloat16:
            b = b.to(torch.bfloat16)
        assert torch.equal(a, b), f"{name}: max |diff| {(a.float() - b.float()).abs().max().item()}"


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,n,transposed", INT64_SHAPES)
def test_column_beyond_2_31_elements(S, B, n, transposed):
    """bf16 Column calls whose (S, B, n) activations have more than 2^31 elements, against the same restatement run in fp64
    torch on the device, chunked over rows.  Every element of every activation output is compared: bf16 outputs to one bf16
    ulp (2^-8 of the value, plus 1e-5 of the chunk's largest), fp32 outputs and the parameter side at COLUMN_TOL."""
    from oracle import oracle as O
    D = _dim(n)
    assert S * B * n > 1 << 31
    gen = torch.Generator(device=dev()).manual_seed(S + n)
    rng = np.random.default_rng(n)
    mu, rho, s1, s2 = (_randn(rng, D) for _ in range(4))
    eps = _randn(rng, S, D)
    bias = _randn(rng, 1 if transposed else n)
    bf = torch.bfloat16
    if transposed:
        x = torch.randn((S, B, n), generator=gen, device=dev(), dtype=bf)
        dy = torch.randn((S, B, 1), generator=gen, device=dev())
    else:
        x = torch.randn((S, B, 1), generator=gen, device=dev(), dtype=bf)
        dy = torch.randn((S, B, n), generator=gen, device=dev(), dtype=bf)
    got = _run_column(x, dy, t(mu), t(rho), t(eps), t(s1), t(s2), t(bias), S, B, n, transposed, False, True)
    g = O.reparam(mu, rho, eps)
    hg, w = _column_weights(g, s1, s2, n)
    _close(got["g"], g, "g", COLUMN_TOL["g"])
    _close(got["hg"], hg, "hg", COLUMN_TOL["hg"])
    wd, bd = torch.tensor(w, device=dev()), torch.tensor(bias, device=dev())
    dwp = torch.zeros((S, n), dtype=torch.float64, device=dev())
    dbias = torch.zeros(bias.shape, dtype=torch.float64, device=dev())
    rows = max(1, (1 << 26) // n)

    def bf16_close(out, ref, what):
        bad = ((out.double() - ref).abs() > 2.0 ** -8 * ref.abs() + 1e-5 * ref.abs().max()).sum().item()
        assert bad == 0, f"{what}: {bad} elements off by more than one bf16 ulp"

    y_err = y_max = 0.0
    for s in range(S):
        for b0 in range(0, B, rows):
            b1 = min(B, b0 + rows)
            xc, dyc = x[s, b0:b1].double(), dy[s, b0:b1].double()
            if transposed:
                yr = xc @ wd[s] + bd[0]
                y_err = max(y_err, (got["y"][s, b0:b1, 0].double() - yr).abs().max().item())
                y_max = max(y_max, yr.abs().max().item())
                bf16_close(got["dx"][s, b0:b1], dyc * wd[s], f"dx s={s} rows {b0}:{b1}")
                dwp[s] += dyc[:, 0] @ xc
                dbias += dyc.sum()
            else:
                bf16_close(got["y"][s, b0:b1], xc * wd[s] + bd, f"y s={s} rows {b0}:{b1}")
                bf16_close(got["dx"][s, b0:b1, 0], dyc @ wd[s], f"dx s={s} rows {b0}:{b1}")
                dwp[s] += xc[:, 0] @ dyc
                dbias += dyc.sum(0)
    if transposed:
        assert y_err <= COLUMN_TOL["y"] * y_max, f"y: rel err {y_err / y_max:.3e}"
    ref = _column_bwd_params(dwp.cpu().numpy(), hg, s1, s2, rho, eps, n)
    ref.update(dwp=dwp.cpu().numpy(), dbias=dbias.cpu().numpy())
    for name in ("dwp", "dbias", "dhg", "dg", "ds2", "dmu", "drho"):
        _close(got[name], ref[name], name, COLUMN_TOL[name])
    _ds1_close(got["ds1"], ref, "ds1")


# ------------------------------------------------------------------------------------------------- reparameterisation
@pytest.mark.gpu
@pytest.mark.parametrize("S,D", REPARAM_SHAPES)
def test_reparam_vs_fp64(S, D):
    """whvi_reparam_f32 into NaN-filled g; whvi_reparam_bwd_f32 into NaN-filled (dmu, drho), then accumulating onto them."""
    from oracle import oracle as O
    from whvi_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(S * 31 + D)
    mu, rho, eps, dg = _randn(rng, D), _randn(rng, D), _randn(rng, S, D), _randn(rng, S, D)
    mut, rhot, epst, dgt = t(mu), t(rho), t(eps), t(dg)
    g = _nan(S, D)
    _lib.check(L.whvi_reparam_f32(mut.data_ptr(), rhot.data_ptr(), epst.data_ptr(), g.data_ptr(), S, D, 0, _stream()), "reparam")
    _close(g, O.reparam(mu, rho, eps), "g", 1e-5)
    dmu, drho = _nan(D), _nan(D)
    for acc in (0, 1):
        _lib.check(L.whvi_reparam_bwd_f32(rhot.data_ptr(), epst.data_ptr(), dgt.data_ptr(), dmu.data_ptr(), drho.data_ptr(), S, D, 0,
                                          acc, _stream()), "reparam_bwd")
        rmu, rrho = O.reparam_bwd(rho, eps, dg)
        _close(dmu, (1 + acc) * rmu, f"dmu (accumulate {acc})", 1e-5)
        _close(drho, (1 + acc) * rrho, f"drho (accumulate {acc})", 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D,G,pstride", STACKED_REPARAM_SHAPES)
def test_grouped_reparam_vs_fp64(S, B, D, G, pstride):
    """The grouped reparameterisation and its backward, as a Stacked call runs them: G groups of S samples, group k's mu and
    rho at + k param_stride.  g is the forward's output; the backward's dmu, drho (G, D) are checked against O.reparam_bwd of
    the dg the call left in its workspace (the kernel's very input), so the check isolates reparam_diag_bwd_kernel."""
    from oracle import oracle as O
    from whvi_b200 import _lib
    from whvi_b200 import functional as F
    L = _lib.lib()
    rng = np.random.default_rng(S * 3 + G * 7 + D)
    mu, rho, s1, s2 = (_randn(rng, G, pstride) for _ in range(4))
    eps, x, dy = _randn(rng, G, S, D), _randn(rng, S, B, D), _randn(rng, S, B, G * D)
    mut, rhot, s1t, s2t, epst = t(mu), t(rho), t(s1), t(s2), t(eps)
    g, yb, y = _nan(G, S, D), _nan(G, S, B, D), _nan(S, B, G * D)
    _lib.check(L.whvi_stacked_fwd_f32(t(x).data_ptr(), B * D, mut.data_ptr(), rhot.data_ptr(), s1t.data_ptr(), s2t.data_ptr(), pstride,
                                      epst.data_ptr(), None, g.data_ptr(), yb.data_ptr(), y.data_ptr(), S, B, D, G, G * D, 0, _stream()),
               "stacked_fwd")
    for k in range(G):
        _close(g[k], O.reparam(mu[k, :D], rho[k, :D], eps[k]), f"g group {k}", 1e-5)
    nbytes = F._query("whvi_stacked_bwd_workspace_bytes", S, B, D, G, 0)[0]
    ws = _nan(_cdiv(nbytes, 4))
    dmu, drho, ds1, ds2 = (_nan(G, D) for _ in range(4))
    _lib.check(L.whvi_stacked_bwd_f32(t(x).data_ptr(), B * D, t(dy).data_ptr(), g.data_ptr(), rhot.data_ptr(), s1t.data_ptr(),
                                      s2t.data_ptr(), pstride, epst.data_ptr(), None, D, dmu.data_ptr(), drho.data_ptr(), ds1.data_ptr(),
                                      ds2.data_ptr(), None, ws.data_ptr(), nbytes, S, B, D, G, G * D, 0, _stream()), "stacked_bwd")
    off = G * S * B * D   # stacked_bwd_layout (api.cu): dy blocks, then dg (G, S, D) when there is no dx
    dg = ws[off:off + G * S * D].view(G, S, D).double().cpu().numpy()
    assert np.isfinite(dg).all()
    for k in range(G):
        rmu, rrho = O.reparam_bwd(rho[k, :D], eps[k], dg[k])
        _close(dmu[k], rmu, f"dmu group {k}", 1e-5)
        _close(drho[k], rrho, f"drho group {k}", 1e-5)


# ------------------------------------------------------------------------------------------------- KL
@pytest.mark.gpu
@pytest.mark.parametrize("D,G,pstride,mode,grad_scale,accumulate", KL_SHAPES)
def test_kl_vs_fp64(D, G, pstride, mode, grad_scale, accumulate):
    """whvi_kl_f32 (G = 0) and whvi_kl_grouped_f32 against sum_k O.kl(mu_k, rho_k): the value into a NaN-filled scalar, the
    gradients (times grad_scale) into NaN-filled buffers or, accumulating, onto random ones."""
    from oracle import oracle as O
    from whvi_b200 import _lib
    L = _lib.lib()
    lam = 0.75
    Gn = max(G, 1)
    rng = np.random.default_rng(D * 5 + G + mode)
    mu, rho = _randn(rng, Gn, max(pstride, D)), _randn(rng, Gn, max(pstride, D))
    base = _randn(rng, 2, Gn, D) if accumulate else np.zeros((2, Gn, D))
    out = _nan(1)
    grads = t(base) if accumulate else _nan(2, Gn, D)
    mut, rhot = (t(mu), t(rho)) if G else (t(mu[0, :D]), t(rho[0, :D]))
    if G:
        rc = L.whvi_kl_grouped_f32(mut.data_ptr(), rhot.data_ptr(), lam, D, G, pstride, mode, out.data_ptr(), grads[0].data_ptr(),
                                   grads[1].data_ptr(), grad_scale, _stream())
    else:
        rc = L.whvi_kl_f32(mut.data_ptr(), rhot.data_ptr(), lam, D, mode, out.data_ptr(), grads[0].data_ptr(),
                           grads[1].data_ptr(), grad_scale, accumulate, _stream())
    _lib.check(rc, "kl")
    refs = [O.kl(mu[k, :D], rho[k, :D], lam, mode, grads=True) for k in range(Gn)]
    value = sum(r[0] for r in refs)
    assert abs(out.item() - value) <= 1e-5 * abs(value), (out.item(), value)
    ref_grads = base + grad_scale * np.stack([np.stack([r[1] for r in refs]), np.stack([r[2] for r in refs])])
    _close(grads[0], ref_grads[0], "dmu", 1e-5)
    _close(grads[1], ref_grads[1], "drho", 1e-5)


# ------------------------------------------------------------------------------------------------- Adam
U32 = 2.0 ** -24   # unit roundoff of fp32


def _adam_ref_moments(g, m, v, b1, b2, grad_scale):
    """fp64 restatement of torch.optim.Adam's moment updates (exp_avg.lerp_(grad, 1 - b1),
    exp_avg_sq.mul_(b2).addcmul_(grad, grad, 1 - b2)) on the scaled gradient."""
    gi = g * grad_scale
    return m + (1 - b1) * (gi - m), b2 * v + (1 - b2) * gi * gi


def _adam_ref_delta(m, v, lr, b1, b2, eps, step):
    """fp64 restatement of torch.optim.Adam's parameter step from the updated moments."""
    bc1, bc2 = 1 - b1 ** step, 1 - b2 ** step
    return -(lr / bc1) * m / (np.sqrt(v) / np.sqrt(bc2) + eps)


@pytest.mark.gpu
@pytest.mark.parametrize("lr_dev,b1,grad_scale", ADAM_ARGS)
@pytest.mark.parametrize("n", ADAM_SIZES)
def test_adam_step_vs_fp64(n, lr_dev, b1, grad_scale):
    """One whvi_adam_f32 step from random p, g, m, v at each t of ADAM_STEPS.  The moments against fp64 to a few ulp of their
    operands (5 u (|m| + (1 - b1)(|g s| + |m|)) for m, 4.5 u v for v); the parameter update dp = p_new - p against the fp64
    step from the stored moments to 1e-5 |dp| plus the half ulp that storing p_new costs.  p is drawn at the scale of dp, so
    that half ulp is small next to dp.  The host lr is wrong on purpose when lr comes from the device."""
    from whvi_b200 import _lib
    L = _lib.lib()
    b1 = float(np.float32(b1))
    b2, eps, lr = float(np.float32(0.999)), float(np.float32(1e-8)), float(np.float32(1e-3))
    for step in ADAM_STEPS:
        rng = np.random.default_rng(n + step)
        p, g, m, v = lr * _randn(rng, n), _randn(rng, n), 0.1 * _randn(rng, n), 0.01 * np.abs(_randn(rng, n))
        p, m, v = (a.astype(np.float32).astype(np.float64) for a in (p, m, v))   # exactly the kernel's inputs
        pt, gt, mt, vt = t(p), t(g), t(m), t(v)
        stept = torch.tensor([float(step)], device=dev())
        lrt = torch.tensor([lr], device=dev())
        rc = L.whvi_adam_f32(pt.data_ptr(), gt.data_ptr(), mt.data_ptr(), vt.data_ptr(), n, 123.0 if lr_dev else lr,
                             lrt.data_ptr() if lr_dev else None, stept.data_ptr(), b1, b2, eps, grad_scale, _stream())
        _lib.check(rc, "whvi_adam_f32")
        m_got, v_got, p_got = (a.double().cpu().numpy() for a in (mt, vt, pt))
        m_ref, v_ref = _adam_ref_moments(g, m, v, b1, b2, grad_scale)
        gi = np.abs(np.float32(g) * np.float32(grad_scale)).astype(np.float64)
        bad = np.abs(m_got - m_ref) > 5 * U32 * (np.abs(m) + (1 - b1) * (gi + np.abs(m)))
        assert not bad.any(), f"t={step}: exp_avg off at {np.flatnonzero(bad)[:5]}"
        bad = np.abs(v_got - v_ref) > 4.5 * U32 * v_ref
        assert not bad.any(), f"t={step}: exp_avg_sq off at {np.flatnonzero(bad)[:5]}"
        dp_ref = _adam_ref_delta(m_got, v_got, lr, b1, b2, eps, step)
        half_ulp = np.spacing(np.abs(p_got).astype(np.float32)).astype(np.float64) / 2
        bad = np.abs((p_got - p) - dp_ref) > 1e-5 * np.abs(dp_ref) + half_ulp
        assert not bad.any(), f"t={step}: parameter step off at {np.flatnonzero(bad)[:5]}"


@pytest.mark.gpu
@pytest.mark.parametrize("n,tensor_lr", [(1000, False), (400_000, True)])
def test_adam_trajectory_vs_torch_adam(n, tensor_lr):
    """50 FlatAdam steps against torch.optim.Adam(foreach=False) on a noisy quadratic, g = p - target + noise_k: the distance
    travelled agrees to 1e-5 of its largest element."""
    from whvi_b200.optim import FlatAdam, FlatParams
    gen = torch.Generator(device=dev()).manual_seed(n)
    p0 = torch.randn(n, generator=gen, device=dev())
    target = torch.randn(n, generator=gen, device=dev())
    noise = torch.randn((50, n), generator=gen, device=dev())
    a, b = torch.nn.Parameter(p0.clone()), torch.nn.Parameter(p0.clone())
    opt_t = torch.optim.Adam([a], lr=1e-2, foreach=False)
    opt_f = FlatAdam(FlatParams([b]), lr=torch.tensor(1e-2, device=dev()) if tensor_lr else 1e-2)
    for k in range(50):
        a.grad = (a.detach() - target + noise[k]).clone()
        with torch.no_grad():
            b.grad.copy_(b - target + noise[k])
        opt_t.step()
        opt_f.step()
    assert float(opt_f.step_t) == 50
    moved = (a.detach() - p0).double().cpu().numpy()
    _close((b.detach() - p0).double(), moved, "p - p0", 1e-5)


# ------------------------------------------------------------------------------------------------- FlatAdam checkpoints
def test_flat_adam_load_state_dict_restores_the_kernel_buffers_cpu():
    """After load_state_dict the buffers the kernel reads hold the loaded step count and moments, are still the objects
    self.state holds, and a tensor lr keeps its identity with the loaded value; a state of another size is refused."""
    from whvi_b200.optim import FlatAdam, FlatParams
    ps = [torch.nn.Parameter(torch.randn(5)), torch.nn.Parameter(torch.randn(2, 3))]
    src = FlatAdam(FlatParams(ps), lr=0.25)
    with torch.no_grad():
        src.exp_avg.fill_(1.0)
        src.exp_avg_sq.copy_(torch.arange(src.flat.numel, dtype=torch.float32))
        src.step_t.fill_(7.0)
    sd = copy.deepcopy(src.state_dict())
    qs = [torch.nn.Parameter(torch.zeros(5)), torch.nn.Parameter(torch.zeros(2, 3))]
    lr = torch.tensor(1e-3)
    opt = FlatAdam(FlatParams(qs), lr=lr)
    bufs = (opt.step_t, opt.exp_avg, opt.exp_avg_sq)
    opt.load_state_dict(sd)
    assert all(a is b for a, b in zip((opt.step_t, opt.exp_avg, opt.exp_avg_sq), bufs))
    st = opt.state[opt.flat.params[0]]
    assert st["step"] is opt.step_t and st["exp_avg"] is opt.exp_avg and st["exp_avg_sq"] is opt.exp_avg_sq
    assert float(opt.step_t) == 7.0
    assert torch.equal(opt.exp_avg, torch.ones(opt.flat.numel))
    assert torch.equal(opt.exp_avg_sq, torch.arange(opt.flat.numel, dtype=torch.float32))
    assert opt.param_groups[0]["lr"] is lr and float(lr) == 0.25
    small = FlatAdam(FlatParams([torch.nn.Parameter(torch.zeros(3))]), lr=1e-3)
    with pytest.raises(ValueError, match="exp_avg"):
        small.load_state_dict(sd)
    assert float(small.step_t) == 0.0 and small.param_groups[0]["lr"] == 1e-3   # a refused load changes nothing


def _resume_model(seed):
    """The toy regression network of test_optim.py with O(1) weights and no posterior noise (rho = -30: softplus(rho) eps
    vanishes below fp32 rounding of mu), so eager and captured steps see the same draws whatever the generator state."""
    import whvi_b200 as W
    torch.manual_seed(seed)
    net = W.WHVIRegression([W.WHVILinear(3, 16, lambda_=2.0), torch.nn.ReLU(), W.WHVILinear(16, 16, lambda_=2.0),
                            torch.nn.ReLU(), W.WHVILinear(16, 1)], train_samples=4).cuda().train()
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.endswith(("s1", "s2", "g_mu")):
                p.normal_()
            if name.endswith("g_rho"):
                p.fill_(-30.0)
    return net


@pytest.mark.gpu
@pytest.mark.parametrize("captured", [False, True])
def test_flat_adam_resume_is_bit_identical(captured):
    """Train 3 steps, torch.save model and optimizer, load both into a fresh model and optimizer (different initial values),
    train 3 more: the parameters equal those of 6 uninterrupted steps bit for bit.  captured: every run steps through a
    GraphedTrainStep, the resumed one captured before the load."""
    from whvi_b200.graphs import GraphedTrainStep
    from whvi_b200.optim import FlatAdam, FlatParams
    g = torch.Generator(device="cuda").manual_seed(9)
    xs = [torch.randn(32, 3, device="cuda", generator=g) for _ in range(6)]
    ys = [x[:, :1] ** 2 - x[:, 1:2] for x in xs]

    def setup(seed):
        net = _resume_model(seed)
        opt = FlatAdam(FlatParams(net.parameters()), lr=torch.tensor(1e-2, device="cuda"))
        stepper = GraphedTrainStep(net, opt, xs[0], ys[0], n=150) if captured else None
        return net, opt, stepper

    def train(net, opt, stepper, ks):
        for k in ks:
            if stepper is not None:
                stepper(xs[k], ys[k])
            else:
                net.loss(xs[k], ys[k], n=150).backward()
                opt.step()
                opt.zero_grad()

    ref, ref_opt, ref_step = setup(1)
    train(ref, ref_opt, ref_step, range(6))
    first, first_opt, first_step = setup(1)
    train(first, first_opt, first_step, range(3))
    buf = io.BytesIO()
    torch.save({"model": first.state_dict(), "opt": first_opt.state_dict()}, buf)
    resumed, opt, stepper = setup(2)
    buf.seek(0)
    ckpt = torch.load(buf, weights_only=False)
    resumed.load_state_dict(ckpt["model"])
    opt.load_state_dict(ckpt["opt"])
    assert float(opt.step_t) == 3.0
    train(resumed, opt, stepper, range(3, 6))
    assert float(opt.step_t) == 6.0
    for (name, p), q in zip(ref.named_parameters(), resumed.parameters()):
        assert torch.equal(p, q), f"{name}: wrong parameters after the resume, max |diff| {(p - q).abs().max().item()}"
