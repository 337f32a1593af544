"""Convolutional WHVI layers: the patch kernels (whvi_im2col_* / whvi_col2im_*), WHVIConv2d and CNN classifiers.

CPU: output-size arithmetic and weight-shape dispatch, state_dict keys and initial values against WHVILinear(C_in kh kw, C_out),
the PAPER-only and CUDA-only rules, argument validation of the four entry points (no CUDA call) and the shim against ctypes.
GPU: im2col bit for bit against F.unfold in the layer's column order (output pre-filled with NaN), col2im against fp64 F.fold,
the layer's output and every gradient against an fp64 restatement whose filters are the oracle's PAPER weights, sample_filters,
patch rows beyond 65535 and more than 2^31 elements, and a small CNN classifier (training, CUDA graph, predict_proba,
state_dict, reference draw order)."""
import copy
import ctypes
import itertools
import warnings

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import rel_err
from oracle import oracle as O

E_NULL, E_SHAPE, E_ALIGN, E_MODE = -1, -2, -3, -4
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference


def _lib():
    from whvi_b200 import _lib
    return _lib.lib()


def _err():
    return _lib().whvi_last_error().decode()


def dev():
    return torch.device("cuda:0")


def _geom(k, stride, pad, dil):
    kh, kw = (k, k) if isinstance(k, int) else k
    return (kh, kw, stride, stride, pad, pad, dil, dil)


# ------------------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("c_in,k,c_out,kind,ld", [
    (4, 2, 16, "square", 16), (1, 3, 40, "stacked", 16), (16, 3, 32, "stacked", 256), (8, 3, 1, "column_t", 72),
    (1, 1, 5, "column", 1), (3, 3, 32, "stacked", 32)])
def test_shape_dispatch_and_output_size(c_in, k, c_out, kind, ld):
    from whvi_b200 import WHVIConv2d, WHVILinear
    from whvi_b200.weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix
    conv = WHVIConv2d(c_in, c_out, k)
    lin = WHVILinear(c_in * k * k, c_out)
    assert type(conv.weight_submodule) is type(lin.weight_submodule)
    expect = {"square": WHVISquarePow2Matrix, "stacked": WHVIStackedMatrix, "column_t": WHVIColumnMatrix,
              "column": WHVIColumnMatrix}[kind]
    assert isinstance(conv.weight_submodule, expect)
    if kind.startswith("column"):
        assert conv.weight_submodule.transposed == (kind == "column_t")
    assert conv.ld == ld and conv.n_in == c_in * k * k
    assert len(conv.square_blocks()) == len(lin.square_blocks())
    for H, W, stride, pad, dil in itertools.product((7, 12), (5, 9), (1, 2, 3), (0, 1, 2), (1, 2)):
        kk = (k, 3) if k > 1 else k
        c = WHVIConv2d(c_in, c_out, kk, stride=stride, padding=pad, dilation=dil)
        ref = nn.Conv2d(c_in, c_out, kk, stride=stride, padding=pad, dilation=dil)
        if min(c.output_size(H, W)) < 1:
            continue
        assert c.output_size(H, W) == tuple(ref(torch.zeros(1, c_in, H, W)).shape[-2:])


def test_pairs_and_bad_geometry():
    from whvi_b200 import WHVIConv2d
    c = WHVIConv2d(2, 8, (3, 1), stride=(2, 1), padding=(1, 0), dilation=(1, 2))
    assert c.geometry == (3, 1, 2, 1, 1, 0, 1, 2) and c.n_in == 6
    for bad in (dict(kernel_size=0), dict(kernel_size=3, stride=0), dict(kernel_size=3, padding=-1), dict(kernel_size=(3, 3, 3))):
        with pytest.raises(ValueError):
            WHVIConv2d(2, 8, **bad)


@pytest.mark.parametrize("c_in,k,c_out", [(4, 2, 16), (1, 3, 40), (16, 3, 32), (8, 3, 1), (1, 1, 5)])
@pytest.mark.parametrize("covariance", ["diag", "dense"])
def test_state_dict_equals_whvilinear(c_in, k, c_out, covariance):
    from whvi_b200 import WHVIConv2d, WHVILinear
    torch.manual_seed(11)
    lin = WHVILinear(c_in * k * k, c_out, lambda_=0.5, bias=True, covariance=covariance)
    torch.manual_seed(11)
    conv = WHVIConv2d(c_in, c_out, k, lambda_=0.5, bias=True, covariance=covariance)
    a, b = lin.state_dict(), conv.state_dict()
    assert list(a) == list(b)
    for key in a:
        assert torch.equal(a[key], b[key]), key
    conv.load_state_dict(a)   # and the other way round


def test_reference_semantics_and_cpu_tensors_raise():
    from whvi_b200 import WHVIConv2d
    with pytest.raises(ValueError, match="paper"):
        WHVIConv2d(3, 8, 3, semantics="reference")
    conv = WHVIConv2d(3, 8, 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        conv(torch.randn(2, 3, 8, 8))
    with pytest.raises(RuntimeError, match="input must be"):
        conv(torch.randn(2, 4, 8, 8))


def _im2col_args(**kw):
    a = dict(x=A, xs=0, out=A, S=2, B=3, H=8, W=9, C=4, kh=3, kw=3, sh=1, sw=1, ph=1, pw=1, dh=1, dw=1, ld=36, st=None)
    a.update(kw)
    return tuple(a.values())


def _col2im_args(**kw):
    a = dict(dp=A, ld=36, dx=A, S=2, B=3, H=8, W=9, C=4, kh=3, kw=3, sh=1, sw=1, ph=1, pw=1, dh=1, dw=1, flags=0, st=None)
    a.update(kw)
    return tuple(a.values())


_VALIDATION = [
    ("im2col", dict(H=2, ph=0), E_SHAPE, "Ho or Wo"),                   # kernel larger than the image: Ho <= 0
    ("im2col", dict(W=4, pw=0, dw=2), E_SHAPE, "Ho or Wo"),
    ("im2col", dict(ld=35), E_SHAPE, "n_in"),
    ("im2col", dict(C=0), E_SHAPE, "[1, 2^24)"),
    ("im2col", dict(sh=0), E_SHAPE, "[1, 2^24)"),
    ("im2col", dict(ph=-1), E_SHAPE, "padding"),
    ("im2col", dict(S=-1), E_SHAPE, "S=-1"),
    ("im2col", dict(xs=5), E_SHAPE, "x_sample_stride"),
    ("im2col", dict(x=None), E_NULL, "null"),
    ("im2col", dict(out=None), E_NULL, "null"),
    ("im2col", dict(x=A + 1), E_ALIGN, "aligned"),
    ("im2col", dict(S=0), 0, ""),                                       # nothing to do: no launch
    ("col2im", dict(ld=35), E_SHAPE, "n_in"),
    ("col2im", dict(H=2, ph=0), E_SHAPE, "Ho or Wo"),
    ("col2im", dict(flags=2), E_MODE, "flags"),
    ("col2im", dict(dx=None), E_NULL, "null"),
    ("col2im", dict(dp=A + 1), E_ALIGN, "aligned"),
    ("col2im", dict(B=0), 0, ""),
]


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_entry_points_validate_without_a_gpu(dtype):
    L = _lib()
    for kind, kw, rc, msg in _VALIDATION:
        args = _im2col_args(**kw) if kind == "im2col" else _col2im_args(**kw)
        got = getattr(L, f"whvi_{kind}_{dtype}")(*args)
        assert got == rc, (kind, kw, got, _err())
        if rc:
            assert msg in _err(), (kind, kw, _err())


def test_shim_and_ctypes_agree():
    L = _lib()
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    for dtype in ("f32", "bf16"):
        for kind, kw, rc, _ in _VALIDATION:
            if rc == 0:
                continue
            name = f"whvi_{kind}_{dtype}"
            fast = getattr(L, name)
            assert not hasattr(fast, "argtypes"), name
            args = _im2col_args(**kw) if kind == "im2col" else _col2im_args(**kw)
            rc_fast, msg_fast = fast(*args), L.whvi_last_error()
            rc_raw, msg_raw = getattr(L._cdll, name)(*args), L.whvi_last_error()
            assert rc_fast == rc_raw == rc and msg_fast == msg_raw, (name, kw)


# ------------------------------------------------------------------------------------------------------------------ GPU
def _stream():
    return torch.cuda.current_stream().cuda_stream


def _raw_im2col(x_cl, geom, ld, per_sample, samples=3):
    """whvi_im2col_* into a NaN-filled output, so that every element is shown to be written; a shared (B, H, W, C) input is
    gathered for ``samples`` samples."""
    S = x_cl.size(0) if per_sample else samples
    B, H, W, C = x_cl.shape[-4:]
    kh, kw, sh, sw, ph, pw, dh, dw = geom
    Ho, Wo = (H + 2 * ph - dh * (kh - 1) - 1) // sh + 1, (W + 2 * pw - dw * (kw - 1) - 1) // sw + 1
    out = torch.full((S, B * Ho * Wo, ld), float("nan"), dtype=x_cl.dtype, device=x_cl.device)
    name = "whvi_im2col_bf16" if x_cl.dtype == torch.bfloat16 else "whvi_im2col_f32"
    rc = getattr(_lib(), name)(x_cl.data_ptr(), x_cl[0].numel() if per_sample else 0, out.data_ptr(), S, B, H, W, C, *geom, ld, _stream())
    assert rc == 0, _err()
    return out


def _unfold_rows(x_nchw, geom, ld):
    """F.unfold rearranged into the layer's column order: (B Ho Wo, ld), column (i kw + j) C + c, zero columns up to ld."""
    kh, kw, sh, sw, ph, pw, dh, dw = geom
    B, C = x_nchw.shape[:2]
    u = F.unfold(x_nchw, (kh, kw), dilation=(dh, dw), padding=(ph, pw), stride=(sh, sw))
    L_ = u.size(-1)
    u = u.reshape(B, C, kh * kw, L_).permute(0, 3, 2, 1).reshape(B * L_, kh * kw * C)
    return F.pad(u, (0, ld - kh * kw * C))


def _fold_image(dp, geom, B, H, W, C):
    """fp64 adjoint of _unfold_rows: F.fold of the (B Ho Wo, ld) patch gradient -> (B, H, W, C)."""
    kh, kw, sh, sw, ph, pw, dh, dw = geom
    n_in = C * kh * kw
    L_ = dp.size(0) // B
    u = dp[:, :n_in].reshape(B, L_, kh * kw, C).permute(0, 3, 2, 1).reshape(B, n_in, L_)
    return F.fold(u, (H, W), (kh, kw), dilation=(dh, dw), padding=(ph, pw), stride=(sh, sw)).permute(0, 2, 3, 1)


_GEOMS = list(itertools.product([1, 3, 5, (3, 1)], [1, 2], [0, 1, 2], [1, 2]))


@pytest.mark.gpu
@pytest.mark.parametrize("k,stride,pad,dil", _GEOMS)
def test_im2col_bit_identical_to_unfold(k, stride, pad, dil):
    geom = _geom(k, stride, pad, dil)
    H, W, B, S = 11, 9, 3, 2
    g = torch.Generator(device=dev()).manual_seed(_GEOMS.index((k, stride, pad, dil)))
    for C, dtype, per_sample in itertools.product((3, 8, 12), (torch.float32, torch.bfloat16), (False, True)):
        n_in = C * geom[0] * geom[1]
        for ld in (n_in, O.next_pow2(n_in), n_in + 5):
            x = torch.randn((S, B, C, H, W), device=dev(), generator=g).to(dtype)
            x_cl = x.permute(0, 1, 3, 4, 2).contiguous()
            got = _raw_im2col(x_cl if per_sample else x_cl[0], geom, ld, per_sample)
            for s in range(got.size(0)):
                ref = _unfold_rows(x[s if per_sample else 0].float(), geom, ld).to(dtype)
                assert torch.equal(got[s], ref), (C, dtype, per_sample, ld, s)


@pytest.mark.gpu
@pytest.mark.parametrize("k,stride,pad,dil", _GEOMS)
def test_col2im_against_fp64_fold(k, stride, pad, dil):
    from whvi_b200 import functional as WF
    geom = _geom(k, stride, pad, dil)
    H, W, B, S = 11, 9, 3, 3
    kh, kw = geom[:2]
    Ho, Wo = WF.conv_output_size(H, kh, stride, pad, dil), WF.conv_output_size(W, kw, stride, pad, dil)
    g = torch.Generator(device=dev()).manual_seed(7)
    for C in (3, 8, 12):
        n_in = C * kh * kw
        for ld in (n_in, O.next_pow2(n_in)):
            dp = torch.randn((S, B * Ho * Wo, ld), device=dev(), generator=g)
            outs = [WF.col2im_(dp[s], geom, (B, H, W, C)) for s in range(S)]
            for s in range(S):
                ref = _fold_image(dp[s].double().cpu(), geom, B, H, W, C)
                assert rel_err(outs[s].cpu().numpy(), ref.numpy()) <= 1e-6, (C, ld, s)
            assert torch.equal(WF.col2im_(dp[0], geom, (B, H, W, C)), outs[0])     # reproducible
            per = WF.col2im_(dp, geom, (B, H, W, C))                                 # (S, B, H, W, C) in one call
            assert all(torch.equal(per[s], outs[s]) for s in range(S))
            total = outs[0]
            for s in range(1, S):
                total = total + outs[s]
            assert torch.equal(WF.col2im_(dp, geom, (B, H, W, C), sum_samples=True), total)
            # bf16: the fp32 call on the widened gradient, rounded once
            db = dp.to(torch.bfloat16)
            assert torch.equal(WF.col2im_(db[1], geom, (B, H, W, C)), WF.col2im_(db[1].float(), geom, (B, H, W, C)).to(torch.bfloat16))
            assert torch.equal(WF.col2im_(db, geom, (B, H, W, C), sum_samples=True),
                               WF.col2im_(db.float(), geom, (B, H, W, C), sum_samples=True).to(torch.bfloat16))


def _randomise(conv, seed):
    """O(1) parameters (the default init makes s1, s2 ~ 0.01) so the oracle comparison sees every term."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in conv.named_parameters():
            if name.endswith("g_rho"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.3 - 1.0)
            elif name.endswith("g_L"):
                D = p.size(0)
                p.copy_(torch.tril(torch.randn(p.shape, generator=g)) / D + torch.eye(D) * 0.5)
            else:
                p.copy_(torch.randn(p.shape, generator=g))


def _oracle_filters(conv, eps, params):
    """(S, C_out, n_in) fp64 weights of the posterior draws with noise ``eps`` (one (S, D) array per square block), from the
    blocks' fp64 parameters ``params`` (torch leaves): g = mu + softplus(rho) eps or mu + L eps, the PAPER weight
    diag(s1) H diag(g) H diag(s2) per block, stacked and truncated (row 0 for a transposed Column weight).  The dense weights
    are checked against the oracle's ``paper_weight``."""
    from whvi_b200.weights import WHVIColumnMatrix
    blocks = []
    for (s1, s2, mu, sig), e in zip(params, eps):
        D = mu.numel()
        Hm = torch.from_numpy(O.build_H(D))
        e = torch.from_numpy(np.asarray(e, dtype=np.float64))
        g = mu + (e @ torch.tril(sig).T if sig.dim() == 2 else F.softplus(sig) * e)
        Wk = s1[None, :, None] * torch.einsum("ij,sj,jk->sik", Hm, g, Hm) * s2[None, None, :]
        for s in range(g.size(0)):
            ref = O.paper_weight(g[s].detach().numpy(), s1.detach().numpy(), s2.detach().numpy())
            assert np.max(np.abs(Wk[s].detach().numpy() - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref)))
        blocks.append(Wk)
    W = torch.cat(blocks, dim=1)
    w = conv.weight_submodule
    if isinstance(w, WHVIColumnMatrix):   # row 0: a (1, n_in) row when transposed, else the (n_out, 1) column
        return W[:, :1, :conv.n_in] if w.transposed else W[:, 0, :conv.out_channels].unsqueeze(-1)
    return W[:, :conv.out_channels, :conv.n_in]


def _block_params(conv):
    dense = conv.square_blocks()[0].covariance == "dense"
    return [(b.s1, b.s2, b.g_mu, b.g_L if dense else b.g_rho) for b in conv.square_blocks()]


def _torch_filters(conv, W):
    kh, kw = conv.kernel_size
    return W.reshape(W.size(0), conv.out_channels, kh, kw, conv.in_channels).permute(0, 1, 4, 2, 3)


def _bias64(conv):
    b = conv.weight_submodule.bias
    return b.detach().double().cpu().requires_grad_()


_LAYER_CASES = [(4, 2, 16, 1, 0, 1), (1, 3, 40, 1, 1, 1), (16, 3, 32, 2, 1, 1), (8, 3, 1, 1, 2, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("c_in,k,c_out,stride,pad,dil", _LAYER_CASES)
@pytest.mark.parametrize("covariance", ["diag", "dense"])
@pytest.mark.parametrize("per_sample", [False, True])
def test_layer_against_fp64_oracle(c_in, k, c_out, stride, pad, dil, covariance, per_sample):
    """fp32: output and every gradient within 1e-4 of the fp64 restatement.  bf16 (same draws): the output is the fp32 output
    on the widened input rounded once, bit for bit; the parameter gradients are within 1e-4 of the fp64 restatement on the
    widened input and upstream gradient; the output and dx carry bf16 rounding (1/256)."""
    from whvi_b200 import WHVIConv2d
    torch.manual_seed(3)
    conv = WHVIConv2d(c_in, c_out, k, stride=stride, padding=pad, dilation=dil, lambda_=1.0, bias=True, covariance=covariance).to(dev())
    _randomise(conv, 5)
    S, B, H, W = 3, 2, 9, 7
    rng = np.random.default_rng(1)
    eps = [rng.standard_normal((S, b.D)) for b in conv.square_blocks()]
    xshape = (S, B, c_in, H, W) if per_sample else (B, c_in, H, W)
    x32 = torch.from_numpy(rng.standard_normal(xshape)).float()
    Ho, Wo = conv.output_size(H, W)
    dy32 = torch.from_numpy(rng.standard_normal((S, B, c_out, Ho, Wo))).float()

    def run(dtype):
        conv.zero_grad(set_to_none=True)
        for b, e in zip(conv.square_blocks(), eps):
            b.inject_eps(torch.from_numpy(e).float().to(dev()))
        x = x32.to(dev(), dtype).requires_grad_()
        conv.mc_samples = S
        try:
            y = conv(x)
        finally:
            conv.mc_samples = None
        assert y.shape == (S, B, c_out, Ho, Wo)
        assert y[0].is_contiguous(memory_format=torch.channels_last)
        (y.float() * dy32.to(dev(), dtype).float()).sum().backward()
        grads = {n: p.grad.detach().cpu().double().numpy() for n, p in conv.named_parameters()}
        return y.detach(), x.grad.detach().cpu().double().numpy(), grads

    for dtype in (torch.float32, torch.bfloat16):
        xq, dyq = x32.to(dtype).double(), dy32.to(dtype).double()
        params = [tuple(t.detach().double().cpu().requires_grad_() for t in blk) for blk in _block_params(conv)]
        bias = _bias64(conv)
        x64 = xq.clone().requires_grad_()
        filt = _torch_filters(conv, _oracle_filters(conv, eps, params))
        b_out = bias.reshape(-1)[:c_out]
        y64 = torch.stack([F.conv2d(x64[s] if per_sample else x64, filt[s], b_out, stride, pad, dil) for s in range(S)])
        (y64 * dyq).sum().backward()
        ref_grads = {}
        for bi, blk in enumerate(params):
            for name, t in zip(("s1", "s2", "g_mu", "g_L" if covariance == "dense" else "g_rho"), blk):
                ref_grads[(bi, name)] = t.grad.numpy()
        y, dx, grads = run(dtype)
        tol_act = 1e-4 if dtype == torch.float32 else 2e-2
        assert rel_err(y.float().cpu().numpy(), y64.detach().numpy()) <= tol_act, dtype
        assert rel_err(dx, x64.grad.numpy()) <= tol_act, dtype
        assert rel_err(grads["weight_submodule.bias"], bias.grad.numpy()) <= 1e-4, dtype
        names = [n for n in grads if n != "weight_submodule.bias"]
        assert len(names) == len(ref_grads)
        for n in names:
            parts = n.split(".")
            bi = int(parts[-2]) if parts[-2].isdigit() else 0
            assert rel_err(grads[n], ref_grads[(bi, parts[-1])]) <= 1e-4, (dtype, n)
        if dtype == torch.bfloat16:   # bf16 activations: the fp32 layer on the widened input, rounded once (im2col is a copy)
            x_w = x32.to(torch.bfloat16).float()
            for b, e in zip(conv.square_blocks(), eps):
                b.inject_eps(torch.from_numpy(e).float().to(dev()))
            conv.mc_samples = S
            try:
                with torch.no_grad():
                    y_w = conv(x_w.to(dev()))
            finally:
                conv.mc_samples = None
            expect = y_w if c_out == 1 else y_w.to(torch.bfloat16)   # a single output channel stays fp32
            assert torch.equal(y, expect)


@pytest.mark.gpu
@pytest.mark.parametrize("c_in,k,c_out,stride,pad,dil", _LAYER_CASES + [(1, 1, 5, 1, 0, 1)])
@pytest.mark.parametrize("covariance", ["diag", "dense"])
def test_sample_filters_match_oracle_and_forward(c_in, k, c_out, stride, pad, dil, covariance):
    from whvi_b200 import WHVIConv2d
    torch.manual_seed(4)
    conv = WHVIConv2d(c_in, c_out, k, stride=stride, padding=pad, dilation=dil, bias=True, covariance=covariance).to(dev())
    _randomise(conv, 9)
    S = 4
    rng = np.random.default_rng(2)
    eps = [rng.standard_normal((S, b.D)) for b in conv.square_blocks()]
    filt = conv.sample_filters(eps=[torch.from_numpy(e).float().to(dev()) for e in eps]).detach()
    kh, kw = conv.kernel_size
    assert filt.shape == (S, c_out, c_in, kh, kw)
    params = [tuple(t.detach().double().cpu() for t in blk) for blk in _block_params(conv)]
    ref = _torch_filters(conv, _oracle_filters(conv, eps, params))
    assert rel_err(filt.cpu().numpy(), ref.numpy()) <= 1e-4
    # the filters are what the forward applies: torch's conv2d with them gives the layer's output
    x = torch.randn(2, c_in, 10, 8, device=dev())
    for b, e in zip(conv.square_blocks(), eps):
        b.inject_eps(torch.from_numpy(e).float().to(dev()))
    conv.mc_samples = S
    try:
        with torch.no_grad():
            y = conv(x)
    finally:
        conv.mc_samples = None
    b = conv.weight_submodule.bias.detach().double().reshape(-1)
    b = b[:c_out]
    for s in range(S):
        ref_y = F.conv2d(x.double(), filt[s].double(), b, stride, pad, dil)
        assert rel_err(y[s].cpu().numpy(), ref_y.cpu().numpy()) <= 1e-4
    assert conv.sample_filters(3).shape == (3, c_out, c_in, kh, kw)


@pytest.mark.gpu
def test_standalone_one_draw_and_channels_last_input():
    from whvi_b200 import WHVIConv2d
    torch.manual_seed(0)
    conv = WHVIConv2d(8, 24, 3, padding=1).to(dev())
    x = torch.randn(5, 8, 12, 12, device=dev())
    for b in conv.square_blocks():
        b.inject_eps(torch.ones(1, b.D, device=dev()))
    y = conv(x)
    assert y.shape == (5, 24, 12, 12) and y.is_contiguous(memory_format=torch.channels_last)
    for b in conv.square_blocks():
        b.inject_eps(torch.ones(1, b.D, device=dev()))
    assert torch.equal(conv(x.contiguous(memory_format=torch.channels_last)), y)


@pytest.mark.gpu
def test_patch_rows_beyond_65535():
    from whvi_b200 import functional as WF
    geom = _geom(3, 1, 1, 1)
    B, H, W, C = 2, 200, 190, 3   # 76000 patch rows
    x = torch.randn(B, C, H, W, device=dev())
    ld = 32
    got = _raw_im2col(x.permute(0, 2, 3, 1).contiguous(), geom, ld, False)[0]
    assert got.size(0) > 65535
    assert torch.equal(got, _unfold_rows(x, geom, ld))
    dp = torch.randn(got.shape, device=dev())
    ref = _fold_image(dp.double().cpu(), geom, B, H, W, C)
    assert rel_err(WF.col2im_(dp, geom, (B, H, W, C)).cpu().numpy(), ref.numpy()) <= 1e-6


@pytest.mark.gpu
def test_beyond_2_31_elements():
    """bf16 (S, B Ho Wo, ld) patches of 2.35e9 elements: every sample of a shared input's patch matrix, and the sample-summed
    col2im of a gradient that size (int64 indexing on both sides)."""
    from whvi_b200 import functional as WF
    geom = _geom(3, 1, 1, 1)
    B, H, W, C, ld, S = 8, 128, 128, 16, 256, 70
    g = torch.Generator(device=dev()).manual_seed(3)
    x = torch.randn((B, H, W, C), device=dev(), generator=g).to(torch.bfloat16)
    N = B * H * W
    assert S * N * ld > 2 ** 31
    got = _raw_im2col(x, geom, ld, False, samples=S)
    ref = _unfold_rows(x.permute(0, 3, 1, 2).float(), geom, ld).to(torch.bfloat16)
    for s in range(S):   # the output was NaN-filled: equality shows every element written
        assert torch.equal(got[s], ref), s
    dp = got
    dp.normal_(generator=g)
    total = None
    for s in range(S):
        part = WF.col2im_(dp[s].float(), geom, (B, H, W, C))
        total = part if total is None else total + part
    assert torch.equal(WF.col2im_(dp, geom, (B, H, W, C), sum_samples=True), total.to(torch.bfloat16))


# ---------------------------------------------------------------------------------------------------------- networks
def _images(n, seed):
    """Two separable classes of 8 x 8 one-channel images: vertical or horizontal bars, plus noise."""
    g = torch.Generator(device=dev()).manual_seed(seed)
    y = torch.randint(0, 2, (n,), device=dev(), generator=g)
    bars = torch.zeros(2, 8, 8, device=dev())
    bars[0, :, ::2] = 1.0
    bars[1, ::2, :] = 1.0
    x = bars[y] + 0.3 * torch.randn((n, 8, 8), device=dev(), generator=g)
    return x.unsqueeze(1), y


def _cnn(seed=0, pool=True, **kw):
    """Three WHVI layers.  The reference's initialisation (s1, s2 ~ 0.01, mu = 0) scales each layer's output by ~1e-4, so
    the logits of three such layers start at ~1e-12 and the gradients vanish; the test starts from s1, s2 ~ N(0, 1/D) and
    mu ~ N(0, 1) instead (each layer keeps the variance of its input) with little posterior noise."""
    import whvi_b200 as W
    torch.manual_seed(seed)
    mods = [W.WHVIConv2d(1, 8, 3, padding=1, lambda_=1.0, bias=True), nn.ReLU()]
    mods += [nn.MaxPool2d(2)] if pool else [W.WHVIConv2d(8, 8, 3, stride=2, padding=1, lambda_=1.0), nn.ReLU()]
    mods += [W.WHVIConv2d(8, 8, 3, padding=1, lambda_=1.0), nn.ReLU(), nn.Flatten(), W.WHVILinear(128, 2, lambda_=1.0, bias=True)]
    net = W.WHVIClassification(mods, train_samples=2, eval_samples=8, **kw)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.endswith(("s1", "s2")):
                p.normal_(0.0, p.numel() ** -0.5)
            elif name.endswith("g_mu"):
                p.normal_()
            elif name.endswith("g_rho"):
                p.fill_(-5.0)
    return net.to(dev())


@pytest.mark.gpu
@pytest.mark.parametrize("bf16", [False, True])
def test_cnn_classifier_learns(bf16):
    net = _cnn()
    x, y = _images(256, 0)
    if bf16:
        x = x.to(torch.bfloat16)
    opt = torch.optim.Adam(net.parameters(), lr=1e-2)
    mnll = []   # the data term: the KL of N(0, 1) means under a lambda = 1 prior moves slowly
    for _ in range(60):
        loss = net.loss(x, y, n=256)
        opt.zero_grad()
        loss.backward()
        opt.step()
        mnll.append(float(net.current_mnll.detach()))
    assert np.mean(mnll[-5:]) < 0.5 * np.mean(mnll[:5]), mnll
    xt, yt = _images(512, 1)
    p = net.predict_proba(xt.to(x.dtype))
    assert p.shape == (512, 2) and torch.allclose(p.sum(1), torch.ones(512, device=dev()), atol=1e-5)
    err, mnll = net.eval_model(xt.to(x.dtype), yt)
    assert err <= 0.1 and mnll == mnll, (err, mnll)
    out = net(xt[:7].to(x.dtype))
    assert out.shape == (7, 2, 8)


@pytest.mark.gpu
def test_cuda_graph_step_equals_eager_step():
    """Posterior noise off (softplus(-30) ~ 1e-13 next to O(1) means), so both runs see the same weights."""
    from whvi_b200 import FlatAdam, FlatParams
    from whvi_b200.graphs import GraphedTrainStep
    eager = _cnn(pool=False)
    with torch.no_grad():
        for name, p in eager.named_parameters():
            if name.endswith("g_mu"):
                p.normal_()
            if name.endswith("g_rho"):
                p.fill_(-30.0)
    graphed = copy.deepcopy(eager)
    opt_e = FlatAdam(FlatParams(eager.parameters()), lr=1e-2)
    opt_g = FlatAdam(FlatParams(graphed.parameters()), lr=1e-2)
    batches = [_images(32, s) for s in range(3)]
    step = GraphedTrainStep(graphed, opt_g, *batches[0], n=256)
    for it, (x, y) in enumerate(batches):
        loss_e = eager.loss(x, y, n=256)
        loss_e.backward()
        opt_e.step()
        opt_e.zero_grad()
        loss_g = step(x, y)
        assert torch.equal(loss_g.detach(), loss_e.detach()), it
        for (k, pe), pg in zip(eager.named_parameters(), graphed.parameters()):
            assert torch.equal(pg.detach(), pe.detach()), (k, it)


@pytest.mark.gpu
def test_train_model_cuda_graph_on_images():
    from whvi_b200 import FlatAdam, FlatParams
    net = _cnn()
    x, y = _images(256, 0)
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(x, y), batch_size=64, shuffle=False)
    opt = FlatAdam(FlatParams(net.parameters()), lr=torch.tensor(1e-2, device=dev()))
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda _: 1.0)
    net.train_model(loader, opt, sched, epochs1=10, epochs2=10, cuda_graph=True)
    err, mnll = net.eval_model(*_images(512, 1))
    assert err <= 0.1 and mnll == mnll, (err, mnll)


@pytest.mark.gpu
def test_state_dict_round_trip():
    net = _cnn(seed=0)
    other = _cnn(seed=1)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        other.load_state_dict(net.state_dict())
    x, _ = _images(16, 3)
    outs = []
    for m in (net, other):
        m.eval()
        torch.manual_seed(5)
        outs.append(m(x))
    assert torch.equal(outs[0], outs[1])


@pytest.mark.gpu
def test_reference_draw_order_is_block_order():
    """rng_mode="reference" draws randn(D) per (sample, layer, block) in loop order; the batched network given those draws
    computes the same logits."""
    ref = _cnn(rng_mode="reference")
    bat = copy.deepcopy(ref)
    bat.rng_mode = "batched"
    ref.eval()
    bat.eval()
    x, _ = _images(8, 4)
    S = ref.eval_samples
    blocks = [b for layer in bat._whvi_layers() for b in layer.square_blocks()]
    assert sum(isinstance(layer, type(ref.sequential[0])) for layer in ref._whvi_layers()) == 2
    torch.manual_seed(9)
    draws = [[] for _ in blocks]
    for _ in range(S):
        for i, b in enumerate(blocks):
            draws[i].append(torch.randn(b.D, device=dev()))
    for b, d in zip(blocks, draws):
        b.inject_eps(torch.stack(d))
    torch.manual_seed(9)
    assert torch.equal(ref(x), bat(x))
