"""CPU: pin the oracle (oracle/) to the reference's own known answers and to golden
fixtures produced by running the reference itself (tests/golden/make_golden.py)."""
import numpy as np
import pytest

from oracle import oracle as O
from conftest import rel_err


# ---- FWHT ------------------------------------------------------------------------------
def test_fwht_known_answers(golden):
    g = golden("fwht")  # test/walsh.py:12-20
    for dt in (np.float32, np.float64):
        out = O.fwht(g["kat_in"].astype(dt))
        assert np.array_equal(out, g["kat_out_expected"].astype(dt))
    assert np.allclose(g["kat_out_cpp"], g["kat_out_expected"], atol=1e-5)


@pytest.mark.parametrize("D", [4, 32, 64, 1024, 4096])
def test_fwht_matches_reference_cpp_and_python(golden, D):
    g = golden("fwht")
    a = g[f"in_{D}"]
    out = O.fwht(a)
    # same butterfly order as src/fwht/cpp/fwht.cpp:8-18 => bit-identical fp32
    assert np.array_equal(out, g[f"cpp_{D}"])
    assert rel_err(out, g[f"py_{D}"]) < 1e-5
    if D <= 1024:
        assert np.allclose(out, g[f"matmul_{D}"], atol=1e-3)
        assert rel_err(O.fwht(a.astype(np.float64)), g[f"dense64_{D}"]) < 1e-12
        assert rel_err(out, g[f"dense64_{D}"]) < 1e-5


@pytest.mark.parametrize("D", [1, 2, 8, 32])
def test_numpy_restatements_agree(D):
    rng = np.random.default_rng(D)
    a = rng.standard_normal((5, D))
    assert np.allclose(O.fwht(a), O.fwht_dense(a), atol=1e-12)
    assert np.allclose(O.fwht(a), O.fwht_cat(a), atol=1e-12)
    H = O.build_H(D)
    assert np.array_equal(H @ H, D * np.eye(D))


def test_fwht_involution_large():
    rng = np.random.default_rng(0)
    a = rng.standard_normal((3, 1 << 15)).astype(np.float32)
    back = O.fwht(O.fwht(a)) / (1 << 15)
    assert rel_err(back, a) < 1e-5


# ---- KL / MNLL --------------------------------------------------------------------------
def test_kl_matches_reference(golden):
    g = golden("kl")
    for i in range(4):
        D, lam = int(g[f"D_{i}"]), float(g[f"lam_{i}"])
        v, dmu, drho = O.kl(g[f"mu_{i}"].astype(np.float64), g[f"rho_{i}"].astype(np.float64), lam, 0, grads=True)
        assert abs(v - float(g[f"kl_{i}"])) <= 2e-5 * max(1.0, abs(v))
        assert rel_err(dmu, g[f"dmu_{i}"]) < 1e-5
        assert rel_err(drho, g[f"drho_{i}"]) < 1e-5
        assert D == g[f"mu_{i}"].shape[0]
    # the reference's formula equals torch's MVN(mu, diag(sd)) KL (test/utils.py:22-34)
    assert np.allclose(g["gen_kl"], g["gen_kl_torch"])


def test_dense_kl_restatement():
    """The dense-covariance KL (not in the reference, "parity unpinned") is tied to pinned things: with L = diag(sigma)
    it is the oracle's sigma^2-form diagonal KL, and for a full L it is torch's closed-form MVN KL (the check the
    reference's test/utils.py:22-34 makes for the diagonal formula); its gradients are its own finite differences."""
    import torch
    rng = np.random.default_rng(5)
    D, lam = 24, 0.37
    mu, rho = rng.standard_normal(D), rng.standard_normal(D) - 1.0
    sigma = np.log1p(np.exp(rho))
    assert abs(O.kl_dense(mu, np.diag(sigma), lam) - O.kl(mu, rho, lam, 1)) < 1e-9 * D
    L = np.tril(rng.standard_normal((D, D))) * 0.3
    L[np.arange(D), np.arange(D)] = np.abs(np.diagonal(L)) + 0.2
    v, dmu, dL = O.kl_dense(mu, L + np.triu(rng.standard_normal((D, D)), 1), lam, grads=True)   # upper part ignored
    q = torch.distributions.MultivariateNormal(torch.tensor(mu), scale_tril=torch.tensor(L))
    p = torch.distributions.MultivariateNormal(torch.zeros(D, dtype=torch.float64), covariance_matrix=lam * torch.eye(D, dtype=torch.float64))
    assert abs(v - torch.distributions.kl_divergence(q, p).item()) < 1e-9 * abs(v)
    h = 1e-6
    for (i, j) in ((0, 0), (5, 2), (23, 23), (7, 7), (2, 5)):
        Lp, Lm = L.copy(), L.copy()
        Lp[i, j] += h
        Lm[i, j] -= h
        fd = (O.kl_dense(mu, Lp, lam) - O.kl_dense(mu, Lm, lam)) / (2 * h)
        assert abs(fd - dL[i, j]) < 1e-5 * max(1.0, abs(fd))
    assert rel_err(dmu, mu / lam) < 1e-12
    dmu_r, dL_r = O.reparam_dense_bwd(rng.standard_normal((3, D)), np.ones((3, D)))
    assert dmu_r.shape == (D,) and np.all(np.triu(dL_r, 1) == 0)


def test_mnll_matches_reference(golden):
    g = golden("mnll")
    assert abs(O.mnll(g["fixed_y"], g["fixed_yhat"], 1.0, 12) - float(g["fixed_mnll"])) < 1e-4
    assert abs(O.mnll(g["rand_y"], g["rand_yhat"], 15.21, 116) - float(g["rand_mnll"])) < 1e-3
    assert abs(O.mnll(g["multi_y"], g["multi_yhat"], 0.7, 40) - float(g["multi_mnll"])) < 1e-3


# ---- reference-as-written layer -------------------------------------------------------
def test_ref_as_written_square(golden):
    g = golden("layers")
    name = "square16"
    x = g[f"{name}.x"].astype(np.float64)
    P = {k: g[f"{name}.param.weight_submodule.{k}"].astype(np.float64) for k in ("s1", "s2", "g_mu", "g_rho")}
    assert int(g[f"{name}.n_eps"]) == 1
    eps = g[f"{name}.eps0"].astype(np.float64)
    sig = O.softplus(P["g_rho"])
    y = O.ref_sample_lrt(x, P["g_mu"], sig * eps, P["s1"], P["s2"])
    assert rel_err(y, g[f"{name}.y"]) < 1e-5
    # SURVEY F1: as written, W collapses to D*diag(s1*g*s2)
    D = 16
    closed = x * (D * P["s1"] * (P["g_mu"] + sig * eps) * P["s2"])
    assert rel_err(closed, g[f"{name}.y"]) < 1e-5
    W = O.ref_w_bar(P["g_mu"], P["s1"], P["s2"])
    assert np.allclose(W, np.diag(D * P["s1"] * P["g_mu"] * P["s2"]), atol=1e-12)


# ---- PAPER layer -------------------------------------------------------------------------
@pytest.mark.parametrize("idx", [0, 1, 2])
def test_paper_layer_matches_dense_autograd(golden, idx):
    g = golden("paper")
    x, s1, s2, mu, rho, eps, dy = (g[f"{k}_{idx}"] for k in ("x", "s1", "s2", "mu", "rho", "eps", "dy"))
    gg = O.reparam(mu, rho, eps)
    assert rel_err(gg, g[f"g_{idx}"]) < 1e-12
    y = O.layer_fwd(x, gg, s1, s2)
    assert rel_err(y, g[f"y_{idx}"]) < 1e-11
    dx, dg, ds1, ds2 = O.layer_bwd(x, dy, gg, s1, s2)
    assert rel_err(dx, g[f"dx_{idx}"]) < 1e-11
    assert rel_err(dg, g[f"dg_{idx}"]) < 1e-11
    assert rel_err(ds1, g[f"ds1_{idx}"]) < 1e-11
    assert rel_err(ds2, g[f"ds2_{idx}"]) < 1e-11
    dmu, drho = O.reparam_bwd(rho, eps, dg)
    assert rel_err(dmu, g[f"dmu_{idx}"]) < 1e-11
    assert rel_err(drho, g[f"drho_{idx}"]) < 1e-11
    # fp32 oracle (the CPU baseline flavour) stays within the layer tolerance
    y32 = O.layer_fwd(x.astype(np.float32), gg.astype(np.float32), s1.astype(np.float32), s2.astype(np.float32))
    assert rel_err(y32, g[f"y_{idx}"]) < 1e-4


def test_paper_dense_weight_and_column():
    rng = np.random.default_rng(5)
    D = 32
    g_, s1, s2 = rng.standard_normal(D), rng.standard_normal(D), rng.standard_normal(D)
    H = O.build_H(D)
    W = np.diag(s1) @ H @ np.diag(g_) @ H @ np.diag(s2)
    assert np.allclose(O.paper_weight(g_, s1, s2), W, atol=1e-10)
    assert np.allclose(O.column_weight_paper(g_, s1, s2, 20), W.reshape(-1)[:20], atol=1e-10)
    x = rng.standard_normal((3, D))
    assert np.allclose(O.layer_fwd(x, g_[None], s1, s2)[0], x @ W.T, atol=1e-9)


def test_shared_x_and_bias():
    rng = np.random.default_rng(6)
    S, B, D = 3, 4, 16
    x = rng.standard_normal((B, D))
    g_, s1, s2, bias = rng.standard_normal((S, D)), rng.standard_normal(D), rng.standard_normal(D), rng.standard_normal(D)
    y_shared = O.layer_fwd(x, g_, s1, s2, bias)
    y_full = O.layer_fwd(np.broadcast_to(x, (S, B, D)).copy(), g_, s1, s2, bias)
    assert np.array_equal(y_shared, y_full)
    dy = rng.standard_normal((S, B, D))
    dx_s, dg_s, ds1_s, ds2_s, db = O.layer_bwd(x, dy, g_, s1, s2, want_dbias=True)
    dx_f, dg_f, ds1_f, ds2_f = O.layer_bwd(np.broadcast_to(x, (S, B, D)).copy(), dy, g_, s1, s2)
    assert np.allclose(dx_s, dx_f.sum(0)) and np.allclose(dg_s, dg_f) and np.allclose(ds1_s, ds1_f)
    assert np.allclose(db, dy.sum((0, 1)))


def test_stacked_dims_match_reference_probe():
    # SURVEY Appendix C probe of WHVIStackedMatrix.setup_dimensions
    assert O.stacked_dims(3, 16) == (4, 16, 1, 4)
    assert O.stacked_dims(13, 128) == (16, 128, 3, 8)
    assert O.stacked_dims(13, 32) == (16, 32, 3, 2)
    assert O.stacked_dims(8, 20) == (8, 24, 0, 3)


def test_oracle_backward_is_the_derivative_of_its_forward():
    """Independent of the reference's autograd goldens: central finite differences (fp64) of the
    oracle's own forward reproduce every gradient its backward returns (layer, reparameterisation, KL)."""
    rng = np.random.default_rng(42)
    S, B, D = 3, 4, 16
    x, g = rng.standard_normal((S, B, D)), rng.standard_normal((S, D))
    s1, s2, bias = rng.standard_normal(D), rng.standard_normal(D), rng.standard_normal(D)
    dy = rng.standard_normal((S, B, D))
    f = lambda x_, g_, s1_, s2_, b_: float((O.layer_fwd(x_, g_, s1_, s2_, b_) * dy).sum())
    dx, dg, ds1, ds2, db = O.layer_bwd(x, dy, g, s1, s2, want_dbias=True)
    h = 1e-6

    def fd(arr, idx, which):
        p, m = arr.copy(), arr.copy()
        p[idx] += h
        m[idx] -= h
        args_p = {"x": x, "g": g, "s1": s1, "s2": s2, "b": bias}
        args_m = dict(args_p)
        args_p[which], args_m[which] = p, m
        return (f(args_p["x"], args_p["g"], args_p["s1"], args_p["s2"], args_p["b"]) -
                f(args_m["x"], args_m["g"], args_m["s1"], args_m["s2"], args_m["b"])) / (2 * h)

    for arr, grad, which in ((x, dx, "x"), (g, dg, "g"), (s1, ds1, "s1"), (s2, ds2, "s2"), (bias, db, "b")):
        for _ in range(6):
            idx = tuple(int(rng.integers(0, n)) for n in arr.shape)
            num = fd(arr, idx, which)
            assert abs(num - grad[idx]) < 1e-6 * max(1.0, abs(num)), (which, idx, num, grad[idx])
    # shared x: dx is summed over the samples
    xs = x[0]
    dxs = O.layer_bwd(xs, dy, g, s1, s2)[0]
    assert rel_err(dxs, O.layer_bwd(np.broadcast_to(xs, (S, B, D)).copy(), dy, g, s1, s2)[0].sum(0)) < 1e-12
    # reparameterisation: g = mu + softplus(rho) * eps
    mu, rho, eps = rng.standard_normal(D), rng.standard_normal(D), rng.standard_normal((S, D))
    w = rng.standard_normal((S, D))
    dmu, drho = O.reparam_bwd(rho, eps, w)
    for j in (0, 5, D - 1):
        rp, rm = rho.copy(), rho.copy()
        rp[j] += h
        rm[j] -= h
        num = float(((O.reparam(mu, rp, eps) - O.reparam(mu, rm, eps)) * w).sum()) / (2 * h)
        assert abs(num - drho[j]) < 1e-6 * max(1.0, abs(num))
        assert abs(dmu[j] - w[:, j].sum()) < 1e-12
    # KL value and gradients, both modes
    for mode in (0, 1):
        val, kmu, krho = O.kl(mu, rho, 1.7, mode, grads=True)
        for j in (1, D - 2):
            for arr, grad, pos in ((mu, kmu, 0), (rho, krho, 1)):
                p, m = arr.copy(), arr.copy()
                p[j] += h
                m[j] -= h
                a = O.kl(p, rho, 1.7, mode) if pos == 0 else O.kl(mu, p, 1.7, mode)
                b = O.kl(m, rho, 1.7, mode) if pos == 0 else O.kl(mu, m, 1.7, mode)
                num = (float(a) - float(b)) / (2 * h)
                assert abs(num - grad[j]) < 1e-6 * max(1.0, abs(num)), (mode, pos, j)


def test_reference_restatement_is_the_reference_layer(golden):
    """The torch restatement (oracle/ref_torch.py) of src/weights.py:66-93, which bench.py's CPU baseline times when the
    reference's own code is not built, reproduces what the reference's own WHVILinear(16, 16) computed
    (tests/golden/layers.npz) on the same parameters and noise: the output and every gradient of its backward.
    Tolerance: fp32 rounding.  The same op sequence on the same host gives identical bits, but the stored values come
    from one host's BLAS.  The restatement evaluated in float64 (inputs and the cached H both cast) lies within
    2.3e-7 of them in this norm (largest: the s1 gradient, 2.23e-7)."""
    import torch
    from oracle import ref_torch
    g = golden("layers")
    t = lambda k: torch.from_numpy(g[f"square16.{k}"])
    assert int(g["square16.n_eps"]) == 1
    x = t("x").requires_grad_()
    P = {k: t(f"param.weight_submodule.{k}").requires_grad_() for k in ("s1", "s2", "g_mu", "g_rho")}
    y = ref_torch.sample_lrt(x, P["s1"], P["s2"], P["g_mu"], P["g_rho"], t("eps0"))
    assert rel_err(y.detach(), g["square16.y"]) < 1e-6
    (y * t("dy")).sum().backward()
    assert rel_err(x.grad, g["square16.dx"]) < 1e-6
    for k, p in P.items():
        assert rel_err(p.grad, g[f"square16.grad.weight_submodule.{k}"]) < 1e-6, k
