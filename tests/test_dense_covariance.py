"""Full-covariance (dense) WHVI posterior for every WHVILinear shape: g = mu + L eps per square block, L lower triangular.

CPU: argument validation of the grouped dense and g-in / dg-out entry points (no CUDA call), the shim against ctypes,
state_dict keys and the initial L.  GPU: the small-D kernels and the grouped KL against the fp64 oracle, the grouped calls at
D >= 128 against the single-block tcgen05 calls, the g-in Stacked / Column calls against the diagonal entry points, module
and network equivalences, CUDA-graph and FlatAdam steps, and the MC evaluation of networks that end in a dense layer."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn

from conftest import rel_err
from oracle import oracle as O

E_NULL, E_SHAPE, E_ALIGN, E_MODE, E_WS = -1, -2, -3, -4, -5
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference


def _lib():
    from whvi_b200 import _lib
    return _lib.lib()


def _err():
    return _lib().whvi_last_error().decode()


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_dense_entry_points_validate_without_a_gpu():
    L = _lib()
    a = A
    f1 = ctypes.c_float(1.0)
    ws = ctypes.c_size_t(0)
    assert L.whvi_reparam_dense_grouped_workspace_bytes(4, 96, ctypes.byref(ws)) == E_SHAPE and "multiple of 128" in _err()
    assert L.whvi_reparam_dense_grouped_workspace_bytes(4, 640, ctypes.byref(ws)) == 0 and ws.value > 0
    assert L.whvi_reparam_dense_grouped_workspace_bytes(4, 64, None) == E_NULL
    assert L.whvi_reparam_dense_grouped_workspace_bytes(4, 64, ctypes.byref(ws)) == 0 and ws.value == 0
    assert L.whvi_reparam_dense_grouped_workspace_bytes(300, 256, ctypes.byref(ws)) == 0 and ws.value > 0
    # reparameterisation: shape, strides, pointers, alignment, workspace
    assert L.whvi_reparam_dense_grouped_f32(a, 96, a, 96 * 96, a, a, 3, 96, 2, None, 0, None) == E_SHAPE
    assert L.whvi_reparam_dense_grouped_f32(a, 8, a, 256, a, a, 3, 16, 2, None, 0, None) == E_SHAPE and "mu_stride" in _err()
    assert L.whvi_reparam_dense_grouped_f32(a, 16, a, 100, a, a, 3, 16, 2, None, 0, None) == E_SHAPE and "L_stride" in _err()
    assert L.whvi_reparam_dense_grouped_f32(a, 130, a, 128 * 128 + 2, a, a, 3, 128, 2, a, 1 << 30, None) == E_SHAPE
    assert L.whvi_reparam_dense_grouped_f32(None, 16, a, 256, a, a, 3, 16, 2, None, 0, None) == E_NULL
    assert L.whvi_reparam_dense_grouped_f32(a, 128, a + 4, 128 * 128, a, a, 3, 128, 1, a, 1 << 30, None) == E_ALIGN
    assert L.whvi_reparam_dense_grouped_f32(a, 128, a, 128 * 128, a, a, 3, 128, 1, a, 16, None) == E_WS and "workspace" in _err()
    assert L.whvi_reparam_dense_grouped_f32(a, 16, a, 256, a, a, 0, 16, 2, None, 0, None) == 0        # S = 0: nothing to do
    # backward
    assert L.whvi_reparam_dense_grouped_bwd_f32(a, a, a, a, -1, 16, 2, None, 0, None) == E_SHAPE
    assert L.whvi_reparam_dense_grouped_bwd_f32(a, a, None, a, 3, 16, 2, None, 0, None) == E_NULL
    assert L.whvi_reparam_dense_grouped_bwd_f32(None, a, a, a, 3, 16, 2, None, 0, None) == E_NULL
    assert L.whvi_reparam_dense_grouped_bwd_f32(a, a, a, a + 4, 3, 256, 2, a, 1 << 30, None) == E_ALIGN
    assert L.whvi_reparam_dense_grouped_bwd_f32(a, a, a, a, 3, 256, 2, a, 64, None) == E_WS
    # grouped KL
    assert L.whvi_kl_dense_grouped_f32(a, 16, a, 256, ctypes.c_float(-1.0), 16, 2, a, None, None, f1, a, 256, None) == E_SHAPE
    assert L.whvi_kl_dense_grouped_f32(a, 16, a, 100, f1, 16, 2, a, None, None, f1, a, 256, None) == E_SHAPE
    assert L.whvi_kl_dense_grouped_f32(a, 16, a, 256, f1, 16, 2, a, a, None, f1, a, 256, None) == E_NULL and "both" in _err()
    assert L.whvi_kl_dense_grouped_f32(a, 16, a, 256, f1, 16, 2, a, None, None, f1, a, 255, None) == E_WS
    assert L.whvi_kl_dense_grouped_f32(a, 16, a, 256, f1, 16, 2, None, None, None, f1, a, 256, None) == E_NULL
    # Stacked from g
    assert L.whvi_stacked_fwd_g_f32(a, 0, a, a, a, 8, None, a, a, 2, 3, 16, 4, 64, 0, None) == E_SHAPE and "param_stride" in _err()
    assert L.whvi_stacked_fwd_g_f32(a, 0, a, a, a, 16, None, a, a, 2, 3, 16, 4, 100, 0, None) == E_SHAPE
    assert L.whvi_stacked_fwd_g_f32(a, 0, a, a, a, 16, None, a, a, 2, 3, 16, 4, 64, 2, None) == E_MODE
    assert L.whvi_stacked_fwd_g_f32(a, 0, None, a, a, 16, None, a, a, 2, 3, 16, 4, 64, 0, None) == E_NULL
    assert L.whvi_stacked_fwd_g_f32(a, 0, a + 4, a, a, 16, None, a, a, 2, 3, 16, 4, 64, 0, None) == E_ALIGN
    assert L.whvi_stacked_bwd_g_f32(a, 0, a, a, a, a, 16, a, 17, a, a, a, None, a, 1 << 30, 2, 3, 16, 4, 64, 0, None) == E_SHAPE
    assert L.whvi_stacked_bwd_g_f32(a, 0, a, a, a, a, 16, None, 13, None, a, a, None, a, 1 << 30, 2, 3, 16, 4, 64, 0, None) == E_NULL
    assert L.whvi_stacked_bwd_g_f32(a, 0, a, a, a, a, 16, None, 13, a, a, a, None, a, 16, 2, 3, 16, 4, 64, 0, None) == E_WS
    # Column from g
    assert L.whvi_column_fwd_g_f32(a, 0, a, a, a, None, a, a, 2, 3, 16, 5, 1, 0, None) == E_SHAPE
    assert L.whvi_column_fwd_g_f32(a, 0, a, a, a, None, a, a, 2, 3, 16, 16, 1, 1, None) == E_MODE and "RELU_OUT" in _err()
    assert L.whvi_column_fwd_g_f32(a, 0, a + 4, a, a, None, a, a, 2, 3, 16, 16, 0, 0, None) == E_ALIGN
    assert L.whvi_column_bwd_g_f32(a, 0, a, a, a, a, None, a, a, a, None, a, 1 << 30, 2, 3, 16, 16, 0, 1, None) == E_MODE
    assert L.whvi_column_bwd_g_f32(a, 0, a, a, a, a, None, None, a, a, None, a, 1 << 30, 2, 3, 16, 16, 1, 0, None) == E_NULL
    assert L.whvi_column_bwd_g_f32(a, 0, a, a, a, a, None, a, a, a, None, a, 16, 2, 3, 16, 16, 1, 0, None) == E_WS


def test_dense_shim_and_ctypes_agree():
    L = _lib()
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    a = A
    cases = [
        ("whvi_reparam_dense_grouped_f32", (a, 8, a, 256, a, a, 3, 16, 2, None, 0, None)),
        ("whvi_reparam_dense_grouped_f32", (a, 128, a, 128 * 128, a, a, 3, 128, 1, a, 16, None)),
        ("whvi_reparam_dense_grouped_bwd_f32", (a, a, None, a, 3, 16, 2, None, 0, None)),
        ("whvi_stacked_fwd_g_f32", (a, 0, a, a, a, 8, None, a, a, 2, 3, 16, 4, 64, 0, None)),
        ("whvi_stacked_bwd_g_f32", (a, 0, a, a, a, a, 16, None, 13, a, a, a, None, a, 16, 2, 3, 16, 4, 64, 0, None)),
        ("whvi_column_fwd_g_f32", (a, 0, a, a, a, None, a, a, 2, 3, 16, 5, 1, 0, None)),
        ("whvi_column_bwd_g_f32", (a, 0, a, a, a, a, None, a, a, a, None, a, 1 << 30, 2, 3, 16, 16, 0, 1, None)),
    ]
    for name, args in cases:
        fast = getattr(L, name)
        assert not hasattr(fast, "argtypes"), name
        rc_fast, msg_fast = fast(*args), L.whvi_last_error()
        rc_raw, msg_raw = getattr(L._cdll, name)(*args), L.whvi_last_error()
        assert rc_fast == rc_raw and rc_fast < 0, (name, rc_fast, rc_raw)
        assert msg_fast == msg_raw and msg_fast, name


@pytest.mark.parametrize("n_in,n_out", [(13, 128), (100, 300), (128, 1), (1, 16), (64, 64)])
def test_dense_state_dict_keys_and_initial_L(n_in, n_out):
    from whvi_b200 import WHVILinear
    torch.manual_seed(7)
    diag = WHVILinear(n_in, n_out, bias=True)
    torch.manual_seed(7)
    dense = WHVILinear(n_in, n_out, bias=True, covariance="dense")
    kd, kx = diag.state_dict(), dense.state_dict()
    rho_keys = [k for k in kd if k.endswith("g_rho")]
    assert rho_keys and not any(k.endswith("g_rho") for k in kx)
    assert sorted(k for k in kx if k.endswith("g_L")) == sorted(k[:-len("g_rho")] + "g_L" for k in rho_keys)
    for k in rho_keys:
        Lk = kx[k[:-len("g_rho")] + "g_L"]
        assert torch.equal(Lk, torch.diag(torch.nn.functional.softplus(kd[k])))
    for k, v in kd.items():
        if not k.endswith("g_rho"):
            assert torch.equal(kx[k], v), k
    with pytest.raises(ValueError):
        WHVILinear(n_in, n_out, semantics="reference", covariance="dense")


# ------------------------------------------------------------------------------------------------------------------ GPU
def dev():
    return torch.device("cuda")


def t(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32, device=dev())


def _grouped_fwd(mu, L, eps):
    """raw whvi_reparam_dense_grouped_f32 on contiguous (G, D) / (G, D, D) / (G, S, D) tensors"""
    from whvi_b200 import functional as WF
    G, S, D = eps.shape
    g = torch.empty_like(eps)
    ws = torch.empty(max(WF._query("whvi_reparam_dense_grouped_workspace_bytes", S, D)[0], 16), dtype=torch.uint8, device=dev())
    rc = _lib().whvi_reparam_dense_grouped_f32(mu.data_ptr(), D, L.data_ptr(), D * D, eps.data_ptr(), g.data_ptr(), S, D, G, ws.data_ptr(),
                                               ws.numel(), None)
    assert rc == 0, _err()
    return g


def _grouped_bwd(eps, dg):
    from whvi_b200 import functional as WF
    G, S, D = eps.shape
    dmu = torch.empty((G, D), device=dev())
    dL = torch.empty((G, D, D), device=dev())
    ws = torch.empty(max(WF._query("whvi_reparam_dense_grouped_workspace_bytes", S, D)[0], 16), dtype=torch.uint8, device=dev())
    rc = _lib().whvi_reparam_dense_grouped_bwd_f32(eps.data_ptr(), dg.data_ptr(), dmu.data_ptr(), dL.data_ptr(), S, D, G, ws.data_ptr(),
                                                   ws.numel(), None)
    assert rc == 0, _err()
    return dmu, dL


def _sum_err(a, b, S):
    """max |a - b| against the size of a sum of S unit-scale terms (sqrt(S)), or of the result where that is larger: a
    heavily cancelled fp32 sum is only as exact as its terms."""
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), np.sqrt(S)))


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 2, 4, 8, 16, 32, 64])
@pytest.mark.parametrize("G", [1, 3, 8])
@pytest.mark.parametrize("S", [1, 37, 300])
def test_small_d_kernels_vs_oracle(D, G, S):
    rng = np.random.default_rng(D * 1000 + G * 10 + S)
    mu = rng.standard_normal((G, D))
    L = rng.standard_normal((G, D, D))          # garbage above the diagonal: ignored
    eps = rng.standard_normal((G, S, D))
    dg = rng.standard_normal((G, S, D))
    g = _grouped_fwd(t(mu), t(L), t(eps))
    dmu, dL = _grouped_bwd(t(eps), t(dg))
    e32, L32, dg32 = eps.astype(np.float32), L.astype(np.float32), dg.astype(np.float32)
    for k in range(G):
        ref_g = O.reparam(mu[k].astype(np.float32).astype(np.float64), np.tril(L32[k]).astype(np.float64), e32[k].astype(np.float64),
                          dense=True)
        assert _sum_err(g[k].cpu().numpy(), ref_g, D) < 1e-5
        rdmu, rdL = O.reparam_dense_bwd(e32[k], dg32[k])
        assert _sum_err(dmu[k].cpu().numpy(), rdmu, S) < 1e-5
        assert _sum_err(dL[k].cpu().numpy(), rdL, S) < 1e-5
        assert np.all(np.triu(dL[k].cpu().numpy(), 1) == 0)
    assert torch.equal(_grouped_fwd(t(mu), t(L), t(eps)), g)
    dmu2, dL2 = _grouped_bwd(t(eps), t(dg))
    assert torch.equal(dmu2, dmu) and torch.equal(dL2, dL)


@pytest.mark.gpu
@pytest.mark.parametrize("D,G", [(16, 8), (64, 3), (128, 3), (1, 2)])
def test_grouped_kl_vs_oracle(D, G):
    from whvi_b200 import functional as WF
    rng = np.random.default_rng(D + G)
    mus = [t(rng.standard_normal(D)).requires_grad_() for _ in range(G)]
    Ls = []
    for _ in range(G):
        L = np.tril(rng.standard_normal((D, D)) * 0.1, -1) + np.diag(rng.uniform(0.5, 1.5, D)) + np.triu(rng.standard_normal((D, D)), 1)
        Ls.append(t(L).requires_grad_())
    lam = 0.3
    kl = WF.kl_gaussian_dense_grouped(mus, Ls, lam)
    kl.backward()
    ref = 0.0
    for k in range(G):
        v, dmu, dL = O.kl_dense(mus[k].detach().cpu().numpy(), Ls[k].detach().cpu().numpy(), lam, grads=True)
        ref += v
        assert rel_err(mus[k].grad.cpu().numpy(), dmu) < 1e-5
        assert rel_err(Ls[k].grad.cpu().numpy(), np.tril(dL)) < 1e-5
    assert abs(kl.item() - ref) < 1e-5 * max(1.0, abs(ref))


@pytest.mark.gpu
@pytest.mark.parametrize("D", [128, 1024])
def test_grouped_large_d_equals_single_block_calls(D):
    from whvi_b200 import functional as WF
    G, S = 3, 37
    rng = np.random.default_rng(D)
    mu, L, eps, dg = (t(rng.standard_normal(s)) for s in ((G, D), (G, D, D), (G, S, D), (G, S, D)))
    g = _grouped_fwd(mu, L, eps)
    dmu, dL = _grouped_bwd(eps, dg)
    lib = _lib()
    for k in range(G):
        gk = torch.empty((S, D), device=dev())
        ws = torch.empty(WF._query("whvi_reparam_dense_workspace_bytes", S, D)[0], dtype=torch.uint8, device=dev())
        assert lib.whvi_reparam_dense_f32(mu[k].data_ptr(), L[k].data_ptr(), eps[k].data_ptr(), gk.data_ptr(), S, D, ws.data_ptr(),
                                          ws.numel(), None) == 0, _err()
        assert torch.equal(g[k], gk)
        Sp = (S + 31) // 32 * 32
        dgT = torch.zeros((D, Sp), device=dev())
        eT = torch.zeros((D, Sp), device=dev())
        dgT[:, :S].copy_(dg[k].t())
        eT[:, :S].copy_(eps[k].t())
        dLk = torch.zeros((D, D), device=dev())
        assert lib.whvi_reparam_dense_bwd_f32(dgT.data_ptr(), eT.data_ptr(), dLk.data_ptr(), Sp, D, None) == 0, _err()
        assert torch.equal(dL[k], dLk)
        assert rel_err(dmu[k].cpu().numpy(), dg[k].sum(0).cpu().numpy()) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("shared,bias,relu", [(True, True, False), (False, False, True), (False, True, True)])
def test_stacked_g_calls_equal_diagonal_entry_points(shared, bias, relu):
    from whvi_b200 import functional as WF
    lib = _lib()
    S, B, D, G, n_in, n_out = 3, 9, 16, 8, 13, 120
    rng = np.random.default_rng(11)
    P = t(rng.standard_normal((G, 4, D)) * 0.5)        # s1, s2, mu, rho per block, param_stride 4 D
    s1, s2, mu, rho = P[:, 0], P[:, 1], P[:, 2], P[:, 3]
    eps = t(rng.standard_normal((G, S, D)))
    x = t(rng.standard_normal((B, D) if shared else (S, B, D)))
    x[..., n_in:] = 0
    xs = 0 if shared else B * D
    bv = t(rng.standard_normal(G * D)) if bias else None
    fl = 1 if relu else 0
    g, yb, y = torch.empty((G, S, D), device=dev()), torch.empty((G, S, B, D), device=dev()), torch.empty((S, B, n_out), device=dev())
    assert lib.whvi_stacked_fwd_f32(x.data_ptr(), xs, mu.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(), 4 * D, eps.data_ptr(),
                                    WF._ptr(bv), g.data_ptr(), yb.data_ptr(), y.data_ptr(), S, B, D, G, n_out, fl, None) == 0, _err()
    y2 = torch.empty_like(y)
    assert lib.whvi_stacked_fwd_g_f32(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), 4 * D, WF._ptr(bv), yb.data_ptr(),
                                      y2.data_ptr(), S, B, D, G, n_out, fl, None) == 0, _err()
    assert torch.equal(y, y2)
    dy = t(rng.standard_normal((S, B, n_out)))
    ws = torch.empty(WF._query("whvi_stacked_bwd_workspace_bytes", S, B, D, G, 1)[0], dtype=torch.uint8, device=dev())
    outs = [torch.empty((5, G, D), device=dev()) for _ in range(2)]
    dxs = [torch.empty((S, B, n_in), device=dev()) for _ in range(2)]
    o, dx = outs[0], dxs[0]
    assert lib.whvi_stacked_bwd_f32(x.data_ptr(), xs, dy.data_ptr(), g.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(), 4 * D,
                                    eps.data_ptr(), dx.data_ptr(), n_in, o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(),
                                    o[4].data_ptr() if bias else None, ws.data_ptr(), ws.numel(), S, B, D, G, n_out, fl, None) == 0, _err()
    o, dx = outs[1], dxs[1]
    dg = torch.empty((G, S, D), device=dev())
    assert lib.whvi_stacked_bwd_g_f32(x.data_ptr(), xs, dy.data_ptr(), g.data_ptr(), s1.data_ptr(), s2.data_ptr(), 4 * D, dx.data_ptr(), n_in,
                                      dg.data_ptr(), o[2].data_ptr(), o[3].data_ptr(), o[4].data_ptr() if bias else None, ws.data_ptr(),
                                      ws.numel(), S, B, D, G, n_out, fl, None) == 0, _err()
    for k in range(G):
        assert lib.whvi_reparam_bwd_f32(rho[k].data_ptr(), eps[k].data_ptr(), dg[k].data_ptr(), o[0, k].data_ptr(), o[1, k].data_ptr(), S,
                                        D, 0, 0, None) == 0, _err()
    assert torch.equal(dxs[0], dxs[1])
    n = 5 if bias else 4
    assert torch.equal(outs[0][:n], outs[1][:n])


@pytest.mark.gpu
@pytest.mark.parametrize("n,transposed,shared,bias", [(128, True, False, True), (16, False, True, True), (100, True, True, False),
                                                      (16, False, False, False)])
def test_column_g_calls_equal_diagonal_entry_points(n, transposed, shared, bias):
    from whvi_b200 import functional as WF
    lib = _lib()
    S, B = 3, 11
    D = 1 << (n - 1).bit_length()
    rng = np.random.default_rng(n)
    mu, rho, s1, s2 = (t(rng.standard_normal(D) * 0.5) for _ in range(4))
    eps = t(rng.standard_normal((S, D)))
    w = n if transposed else 1
    x = t(rng.standard_normal((B, w) if shared else (S, B, w)))
    xs = 0 if shared else B * w
    bv = t(rng.standard_normal(1 if transposed else n)) if bias else None
    ny = 1 if transposed else n
    g, hg, y = torch.empty((S, D), device=dev()), torch.empty((S, D), device=dev()), torch.empty((S, B, ny), device=dev())
    tr = 1 if transposed else 0
    assert lib.whvi_column_fwd_f32(x.data_ptr(), xs, mu.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(), eps.data_ptr(), WF._ptr(bv),
                                   g.data_ptr(), hg.data_ptr(), y.data_ptr(), S, B, D, n, tr, 0, None) == 0, _err()
    hg2, y2 = torch.empty_like(hg), torch.empty_like(y)
    assert lib.whvi_column_fwd_g_f32(x.data_ptr(), xs, g.data_ptr(), s1.data_ptr(), s2.data_ptr(), WF._ptr(bv), hg2.data_ptr(), y2.data_ptr(),
                                     S, B, D, n, tr, 0, None) == 0, _err()
    assert torch.equal(hg, hg2) and torch.equal(y, y2)
    dy = t(rng.standard_normal((S, B, ny)))
    ws = torch.empty(WF._query("whvi_column_bwd_workspace_bytes", S, D, n)[0], dtype=torch.uint8, device=dev())
    outs = [torch.empty((4, D), device=dev()) for _ in range(2)]
    dbs = [torch.empty(ny, device=dev()) if bias else None for _ in range(2)]
    dxs = [torch.empty((S, B, w), device=dev()) for _ in range(2)]
    o = outs[0]
    assert lib.whvi_column_bwd_f32(x.data_ptr(), xs, dy.data_ptr(), hg.data_ptr(), rho.data_ptr(), s1.data_ptr(), s2.data_ptr(), eps.data_ptr(),
                                   dxs[0].data_ptr(), o[0].data_ptr(), o[1].data_ptr(), o[2].data_ptr(), o[3].data_ptr(), WF._ptr(dbs[0]),
                                   ws.data_ptr(), ws.numel(), S, B, D, n, tr, 0, None) == 0, _err()
    o = outs[1]
    dg = torch.empty((S, D), device=dev())
    assert lib.whvi_column_bwd_g_f32(x.data_ptr(), xs, dy.data_ptr(), hg.data_ptr(), s1.data_ptr(), s2.data_ptr(), dxs[1].data_ptr(),
                                     dg.data_ptr(), o[2].data_ptr(), o[3].data_ptr(), WF._ptr(dbs[1]), ws.data_ptr(), ws.numel(), S, B, D, n,
                                     tr, 0, None) == 0, _err()
    assert lib.whvi_reparam_bwd_f32(rho.data_ptr(), eps.data_ptr(), dg.data_ptr(), o[0].data_ptr(), o[1].data_ptr(), S, D, 0, 0, None) == 0
    assert torch.equal(outs[0], outs[1]) and torch.equal(dxs[0], dxs[1])
    if bias:
        assert torch.equal(dbs[0], dbs[1])


def _blocks(layer):
    return layer.square_blocks()


@pytest.mark.gpu
@pytest.mark.parametrize("n_in,n_out", [(13, 128), (100, 300), (128, 1), (1, 16), (64, 64)])
@pytest.mark.parametrize("shared", [True, False])
@pytest.mark.parametrize("bias", [True, False])
def test_dense_module_equals_diagonal_at_diagonal_L(n_in, n_out, shared, bias):
    """Dense with L = diag(softplus(rho)) and the same noise is the diagonal module with the sigma^2 KL (kl_mode=1)."""
    from whvi_b200 import WHVILinear
    S, B = 5, 9
    torch.manual_seed(3)
    a = WHVILinear(n_in, n_out, lambda_=0.1, bias=bias, kl_mode=1).to(dev())
    torch.manual_seed(3)
    b = WHVILinear(n_in, n_out, lambda_=0.1, bias=bias, covariance="dense").to(dev())
    torch.manual_seed(4)
    x = torch.randn(B, n_in, device=dev()) if shared else torch.randn(S, B, n_in, device=dev())
    eps = [torch.randn(S, blk.D, device=dev()) for blk in _blocks(a)]
    outs = []
    for m in (a, b):
        m.mc_samples = S
        for blk, e in zip(_blocks(m), eps):
            blk.inject_eps(e.clone())
        y = m(x)
        kl = m.kl
        (y.square().sum() + (y * 0.3).sum() + kl).backward()
        outs.append((y.detach().cpu().numpy(), kl.item()))
        m.mc_samples = None
    assert rel_err(outs[1][0], outs[0][0]) < 1e-5
    assert abs(outs[1][1] - outs[0][1]) < 1e-5 * abs(outs[0][1])
    for ba, bb in zip(_blocks(a), _blocks(b)):
        for n in ("s1", "s2", "g_mu"):
            assert rel_err(getattr(bb, n).grad.cpu().numpy(), getattr(ba, n).grad.cpu().numpy()) < 1e-4, n
        sig_grad = ba.g_rho.grad / torch.sigmoid(ba.g_rho.detach())
        assert rel_err(torch.diagonal(bb.g_L.grad).cpu().numpy(), sig_grad.cpu().numpy()) < 1e-4
        assert np.all(np.triu(bb.g_L.grad.cpu().numpy(), 1) == 0)
    if bias:
        assert rel_err(b.weight_submodule.bias.grad.cpu().numpy(), a.weight_submodule.bias.grad.cpu().numpy()) < 1e-4


def _randomise_L(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for m in model.modules():
            if getattr(m, "covariance", None) == "dense":
                D = m.D
                m.g_L.add_(torch.tril(torch.randn(D, D, generator=g), -1).to(m.g_L.device) * (0.3 / D ** 0.5))
                m.g_mu.add_(torch.randn(D, generator=g).to(m.g_mu.device) * 0.1)


@pytest.mark.gpu
@pytest.mark.parametrize("n_in,n_out", [(13, 128), (100, 300)])
def test_stacked_grouped_equals_block_by_block_full_L(n_in, n_out):
    import copy
    from whvi_b200 import WHVILinear
    S, B = 4, 7
    torch.manual_seed(1)
    a = WHVILinear(n_in, n_out, lambda_=0.5, bias=True, covariance="dense").to(dev())
    _randomise_L(a, 2)
    b = copy.deepcopy(a)
    b.weight_submodule.one_launch = False
    assert a.weight_submodule.grouped and not b.weight_submodule.grouped
    x = torch.randn(S, B, n_in, device=dev())
    eps = [torch.randn(S, blk.D, device=dev()) for blk in _blocks(a)]
    outs = []
    for m in (a, b):
        m.mc_samples = S
        for blk, e in zip(_blocks(m), eps):
            blk.inject_eps(e.clone())
        xi = x.clone().requires_grad_()
        y = m(xi)
        kl = m.kl
        (y.square().sum() + kl).backward()
        outs.append((y.detach(), kl.detach(), xi.grad))
    assert rel_err(outs[0][0].cpu().numpy(), outs[1][0].cpu().numpy()) < 1e-5
    assert abs(outs[0][1].item() - outs[1][1].item()) < 1e-5 * abs(outs[1][1].item())
    assert rel_err(outs[0][2].cpu().numpy(), outs[1][2].cpu().numpy()) < 1e-4
    for (n, p), q in zip(a.named_parameters(), b.parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) < 1e-4, n


def _config3(dense=True, seed=0):
    from whvi_b200 import WHVILinear, WHVIRegression
    torch.manual_seed(seed)
    cov = "dense" if dense else "diag"
    m = WHVIRegression([WHVILinear(13, 128, covariance=cov), nn.ReLU(), WHVILinear(128, 128, covariance=cov), nn.ReLU(),
                        WHVILinear(128, 1, covariance=cov)], sigma=0.5, train_samples=8).to(dev())
    if dense:
        _randomise_L(m, seed + 1)
    return m


@pytest.mark.gpu
def test_config3_dense_loss_backward_equals_block_by_block():
    import copy
    a = _config3()
    b = copy.deepcopy(a)
    for mod in b.modules():
        if hasattr(mod, "one_launch"):
            mod.one_launch = False
    x = torch.randn(64, 13, device=dev())
    y = torch.randn(64, 1, device=dev())
    S = a.train_samples
    eps = [torch.randn(S, blk.D, device=dev()) for layer in a._whvi_layers() for blk in layer.square_blocks()]
    losses = []
    for m in (a, b):
        m.train()
        for blk, e in zip([blk for layer in m._whvi_layers() for blk in layer.square_blocks()], eps):
            blk.inject_eps(e.clone())
        loss = m.loss(x, y, n=1000)
        loss.backward()
        losses.append(loss.item())
    assert abs(losses[0] - losses[1]) < 1e-4 * abs(losses[1])
    for (n, p), q in zip(a.named_parameters(), b.parameters()):
        if p.grad is not None or q.grad is not None:
            assert rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) < 1e-4, n


@pytest.mark.gpu
def test_config3_dense_cuda_graph_step_matches_eager_and_flat_adam_runs():
    """Fixed injected noise per step: a captured step reads the injected tensors where they lie, so eager and graph replays
    see the same noise."""
    import copy
    from whvi_b200.graphs import GraphedTrainStep
    from whvi_b200.optim import FlatAdam, FlatParams
    gen = torch.Generator(device="cuda").manual_seed(5)
    xs = [torch.randn(32, 13, device="cuda", generator=gen) for _ in range(4)]
    ys = [x[:, :1] ** 2 - x[:, 1:2] for x in xs]
    eager = _config3(seed=9)
    graphed = copy.deepcopy(eager)
    S = eager.train_samples
    E = [torch.randn(S, blk.D, device="cuda", generator=gen) for layer in eager._whvi_layers() for blk in layer.square_blocks()]

    def inject(model, times=1):
        for _ in range(times):
            for blk, e in zip([b for layer in model._whvi_layers() for b in layer.square_blocks()], E):
                blk.inject_eps(e)

    opt_e = torch.optim.Adam(eager.parameters(), lr=torch.tensor(1e-3, device="cuda"), capturable=True)
    opt_g = torch.optim.Adam(graphed.parameters(), lr=torch.tensor(1e-3, device="cuda"), capturable=True)
    eager.train(), graphed.train()
    inject(graphed, 4)   # three warm-up steps and the capture
    step = GraphedTrainStep(graphed, opt_g, xs[0], ys[0], n=150)
    for p, q in zip(eager.parameters(), graphed.parameters()):
        assert torch.equal(p, q)
    losses_e, losses_g = [], []
    for x, y in zip(xs, ys):
        inject(eager)
        loss = eager.loss(x, y, n=150)
        loss.backward()
        opt_e.step()
        opt_e.zero_grad(set_to_none=True)
        losses_e.append(float(loss))
        losses_g.append(float(step(x, y)))
    assert np.allclose(losses_e, losses_g, rtol=1e-4), (losses_e, losses_g)
    for (name, p), q in zip(eager.named_parameters(), graphed.parameters()):
        assert rel_err(q.detach().cpu().numpy(), p.detach().cpu().numpy()) < 1e-4, name
    # FlatAdam over the dense parameters (the Stacked blocks' g_L read where FlatParams puts them)
    m = _config3(seed=13)
    before = [p.detach().clone() for p in m.parameters()]
    L0 = m.sequential[0].weight_submodule.weight_matrices[0].g_L
    L0_before = L0.detach().clone()
    opt = FlatAdam(FlatParams(m.parameters()), lr=torch.tensor(1e-3, device="cuda"))
    m.train()
    for x, y in zip(xs, ys):
        loss = m.loss(x, y, n=150)
        loss.backward()
        opt.step()
        opt.zero_grad()
        assert np.isfinite(float(loss))
    assert any(not torch.equal(p, q) for p, q in zip(m.parameters(), before))
    assert not torch.equal(torch.tril(L0.detach(), -1), torch.tril(L0_before, -1))   # the off-diagonal of L trains too


@pytest.mark.gpu
@pytest.mark.parametrize("D", [256, 8192])
@pytest.mark.parametrize("layers", [1, 2])
def test_eval_model_dense_last_layer_equals_full_prediction(D, layers):
    from whvi_b200 import WHVILinear, WHVIRegression
    torch.manual_seed(D + layers)
    mods = [WHVILinear(D, D, covariance="dense")] if layers == 1 else [WHVILinear(D, D, covariance="dense"), nn.ReLU(),
                                                                       WHVILinear(D, D, covariance="dense")]
    m = WHVIRegression(mods, sigma=0.7, eval_samples=6).to(dev())
    _randomise_L(m, D)
    B = 5
    X = torch.randn(B, D, device=dev())
    y = torch.randn(B, D, device=dev())
    m.eval()
    S = m.eval_samples
    eps = [torch.randn(S, D, device=dev()) for _ in m._whvi_layers()]
    for layer, e in zip(m._whvi_layers(), eps):
        layer.weight_submodule.inject_eps(e.clone())
    sum_y, sum_y2, n = m.predictive_sums(X)
    for layer, e in zip(m._whvi_layers(), eps):
        layer.weight_submodule.inject_eps(e.clone())
    with torch.no_grad():
        pred = m(X)                                      # (B, out, S)
    ref_y, ref_y2 = pred.sum(-1), pred.square().sum(-1)
    assert n == S
    assert rel_err(sum_y.cpu().numpy(), ref_y.cpu().numpy()) < 1e-4
    assert rel_err(sum_y2.cpu().numpy(), ref_y2.cpu().numpy()) < 1e-4
    from whvi_b200.networks import WHVINetwork
    for layer, e in zip(m._whvi_layers(), eps):
        layer.weight_submodule.inject_eps(e.clone())
    rmse, mnll = m.eval_model(X, y)                     # from predictive_sums
    for layer, e in zip(m._whvi_layers(), eps):
        layer.weight_submodule.inject_eps(e.clone())
    rmse_f, mnll_f = WHVINetwork.eval_model(m, X, y, lambda p, t_: torch.sqrt(((p.mean(dim=2) - t_) ** 2).mean()))
    assert abs(rmse - rmse_f) < 1e-4 * abs(rmse_f)
    assert abs(mnll - mnll_f) < 1e-4 * abs(mnll_f)
