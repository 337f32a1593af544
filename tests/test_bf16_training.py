"""Training with bf16 activations: ``whvi_layer_bwd_bf16`` / ``whvi_layer_loss_bf16`` and everything above them.

Definition checked throughout: a bf16 call is the fp32 call on the widened inputs with the same plan, so the parameter
gradients (and the squared-error partial sums) are bit-identical to the fp32 kernels' for float(x), float(dy), and dx is
bf16(dx_f32), rounded once.  The CPU tests check argument validation only; the GPU tests check the definition with
``torch.equal``."""
import ctypes

import pytest
import torch

E_NULL, E_SHAPE, E_ALIGN, E_MODE = -1, -2, -3, -4
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference


def _bwd_args(**kw):
    a = dict(x=A, xs=0, dy=A, dy_scale=None, g=A, s1=A, s2=A, dx=A, dg=A, ds1=A, ds2=A, dbias=None, ws=A, ws_bytes=1 << 30,
             S=2, B=3, D=64, flags=0, stream=None)
    a.update(kw)
    return tuple(a.values())


def _loss_args(**kw):
    a = dict(x=A, xs=0, g=A, s1=A, s2=A, bias=None, target=A, dx=A, dg=A, ds1=A, ds2=A, dbias=None, sqp=A, ws=A,
             ws_bytes=1 << 30, S=2, B=3, D=256, flags=0, stream=None)
    a.update(kw)
    return tuple(a.values())


BWD_CASES = [
    (_bwd_args(D=16384), E_SHAPE, "outside"),                  # the fused backward stops at 8192 (multi-pass above, in Python)
    (_bwd_args(D=2), E_SHAPE, "outside"),
    (_bwd_args(D=48), E_SHAPE, "power of 2"),
    (_bwd_args(xs=7), E_SHAPE, "x_sample_stride"),
    (_bwd_args(D=4, B=5), E_SHAPE, "multiple of 8"),            # bulk-copy granularity: D = 4 with an odd B
    (_bwd_args(flags=2), E_MODE, "unknown flags"),
    (_bwd_args(dg=None), E_NULL, "null output"),
    (_bwd_args(x=None), E_NULL, "null pointer"),
    (_bwd_args(dy=None), E_NULL, "null pointer"),
    (_bwd_args(x=A + 8), E_ALIGN, "x and dy"),                  # bf16 x must still be 16-byte aligned (bulk copies)
    (_bwd_args(dy=A + 8), E_ALIGN, "x and dy"),
    (_bwd_args(dx=A + 4), E_ALIGN, "dx 8-byte"),
    (_bwd_args(g=A + 4), E_ALIGN, "fp32 pointers"),
    (_bwd_args(ws=A + 4), E_ALIGN, "fp32 pointers"),
]
LOSS_CASES = [
    (_loss_args(D=64), E_SHAPE, "outside [128, 4096]"),
    (_loss_args(D=8192), E_SHAPE, "outside"),
    (_loss_args(D=384), E_SHAPE, "power of 2"),
    (_loss_args(B=0), E_SHAPE, "empty batch"),
    (_loss_args(xs=5), E_SHAPE, "x_sample_stride"),
    (_loss_args(flags=4), E_MODE, "unknown flags"),
    (_loss_args(target=None), E_NULL, "null pointer"),
    (_loss_args(bias=A), E_NULL, "null pointer"),               # bias without dbias
    (_loss_args(x=None), E_NULL, "null pointer"),
    (_loss_args(x=A + 8), E_ALIGN, "x must be 16-byte"),
    (_loss_args(dx=A + 2), E_ALIGN, "dx 8-byte"),
    (_loss_args(target=A + 4), E_ALIGN, "fp32 pointers"),
]


def test_bf16_entry_points_validate_before_any_cuda_call():
    from whvi_b200 import _lib
    L = _lib.lib()
    for args, code, msg in BWD_CASES:
        assert L.whvi_layer_bwd_bf16(*args) == code, args
        assert msg in L.whvi_last_error().decode(), (args, L.whvi_last_error())
    for args, code, msg in LOSS_CASES:
        assert L.whvi_layer_loss_bf16(*args) == code, args
        assert msg in L.whvi_last_error().decode(), (args, L.whvi_last_error())
    # the workspace is the fp32 call's (same plan): the fp32 size query serves both
    ws = ctypes.c_size_t(0)
    assert L.whvi_layer_bwd_workspace_bytes(2, 3, 64, ctypes.byref(ws)) == 0 and ws.value > 0


def test_bf16_entry_points_shim_matches_ctypes():
    from whvi_b200 import _lib
    L = _lib.lib()
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    for name, cases in (("whvi_layer_bwd_bf16", BWD_CASES), ("whvi_layer_loss_bf16", LOSS_CASES)):
        fast, raw = getattr(L, name), getattr(L._cdll, name)
        assert not hasattr(fast, "argtypes"), name
        for args, _, _ in cases:
            rc_fast, msg_fast = fast(*args), L.whvi_last_error()
            rc_raw, msg_raw = raw(*args), L.whvi_last_error()
            assert rc_fast == rc_raw < 0 and msg_fast == msg_raw and msg_fast, (name, args)


def test_resid_backward_is_fp32_only():
    """The saved-output + target backward (the sq-err layer's) has no bf16 kernel: asking for it raises, nothing upcasts."""
    from whvi_b200 import functional as F
    x = torch.zeros(2, 3, 8, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="fp32 only"):
        F.layer_backward_raw(x, x, torch.zeros(2, 8), torch.zeros(8), torch.zeros(8), target=torch.zeros(3, 8),
                             coef=torch.ones(1))


def test_unsupported_modules_reject_bf16():
    from whvi_b200.weights import WHVIColumnMatrix, WHVISquarePow2Matrix, WHVIStackedMatrix
    x = torch.zeros(3, 8, dtype=torch.bfloat16)
    with pytest.raises(RuntimeError, match="bf16"):
        WHVIStackedMatrix(8, 24)(x)
    with pytest.raises(RuntimeError, match="bf16"):
        WHVIColumnMatrix(8, transposed=True)(x)
    with pytest.raises(RuntimeError, match="bf16"):
        WHVISquarePow2Matrix(8, semantics="reference")(x)


# ------------------------------------------------------------------------------------------------------------------- GPU
def dev():
    return torch.device("cuda:0")


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(shape, g, dtype=torch.float32):
    return torch.randn(shape, generator=g, device=dev()).to(dtype)


def _eq(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, what
    assert torch.equal(a, b), f"{what}: max |diff| {(a.float() - b.float()).abs().max().item()}"


# (D, S, B): B chosen so that a sample's rows end in a partial tile where D is below the tile (1024 elements for
# D <= 1024, 4096 at 2048 / 4096, 8192 at 8192); D = 4 with B odd takes the zero-row padding.  The large-B cases give every
# tile pair 8 tiles, more than its staging ring holds, so the ring wraps (stage reuse after the empty-barrier wait).
BWD_SHAPES = [(4, 3, 37), (4, 2, 300), (16, 3, 67), (128, 2, 9), (1024, 3, 5), (2048, 2, 3), (4096, 2, 3), (8192, 2, 3),
              (1 << 14, 2, 3), (1 << 15, 2, 2), (1024, 2, 2048), (4096, 2, 512), (8192, 2, 64)]
# (relu_in, dy_scale, want_dx, want_dbias)
BWD_FLAGS = [(False, None, True, True), (True, 0.375, True, False), (True, None, False, True), (False, 1.5, True, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("D,S,B", BWD_SHAPES)
@pytest.mark.parametrize("shared", [False, True])
def test_backward_bf16_is_fp32_on_widened_inputs(D, S, B, shared):
    from whvi_b200 import functional as F
    g = _gen(D + B)
    x = _randn((B, D) if shared else (S, B, D), g, torch.bfloat16)
    dy = _randn((S, B, D), g, torch.bfloat16)
    gs, s1, s2 = _randn((S, D), g), _randn(D, g), _randn(D, g)
    for relu_in, scale, want_dx, want_db in BWD_FLAGS:
        sc = None if scale is None else torch.full((1,), scale, device=dev())
        got = F.layer_backward_raw(x, dy, gs, s1, s2, want_dx=want_dx, want_dbias=want_db, relu_in=relu_in, dy_scale=sc)
        ref = F.layer_backward_raw(x.float(), dy.float(), gs, s1, s2, want_dx=want_dx, want_dbias=want_db, relu_in=relu_in,
                                   dy_scale=sc)
        tag = f"D={D} S={S} B={B} shared={shared} relu_in={relu_in} scale={scale}"
        if want_dx:
            _eq(got[0], ref[0].to(torch.bfloat16), f"dx {tag}")
        else:
            assert got[0] is None
        for name, a, b in zip(("dg", "ds1", "ds2"), got[1:4], ref[1:4]):
            _eq(a, b, f"{name} {tag}")
        if want_db:
            _eq(got[4], ref[4], f"dbias {tag}")
        else:
            assert got[4] is None


@pytest.mark.gpu
@pytest.mark.parametrize("D,S,B", [(128, 3, 9), (1024, 2, 7), (2048, 2, 3), (4096, 2, 5), (1024, 2, 2048), (4096, 2, 512)])
@pytest.mark.parametrize("bias", [False, True])     # at 2048 / 4096: without bias the tensor-memory kernel, with bias the other
@pytest.mark.parametrize("shared", [False, True])
def test_loss_layer_bf16_is_fp32_on_widened_inputs(D, S, B, bias, shared):
    from whvi_b200 import functional as F
    g = _gen(3 * D + B)
    x = _randn((B, D) if shared else (S, B, D), g, torch.bfloat16)
    gs, s1, s2, target = _randn((S, D), g), _randn(D, g), _randn(D, g), _randn((B, D), g)
    b = _randn(D, g) if bias else None
    for relu_in in (False, True):
        got = F.layer_loss_raw(x, gs, s1, s2, b, target, relu_in=relu_in)
        ref = F.layer_loss_raw(x.float(), gs, s1, s2, b, target, relu_in=relu_in)
        tag = f"D={D} S={S} B={B} bias={bias} shared={shared} relu_in={relu_in}"
        _eq(got[0], ref[0], f"sum r^2 {tag}")
        _eq(got[1], ref[1].to(torch.bfloat16), f"dx {tag}")
        for name, a, c in zip(("dg", "ds1", "ds2"), got[2:5], ref[2:5]):
            _eq(a, c, f"{name} {tag}")
        if bias:
            _eq(got[5], ref[5], f"dbias {tag}")


@pytest.mark.gpu
@pytest.mark.parametrize("D,covariance", [(4, "diag"), (256, "diag"), (2048, "diag"), (256, "dense"), (2048, "dense")])
def test_square_module_autograd_bf16(D, covariance):
    """Module forward + autograd: output and x.grad are bf16, parameter gradients fp32 and equal to the raw kernels."""
    from whvi_b200 import functional as F
    from whvi_b200.weights import WHVISquarePow2Matrix
    torch.manual_seed(D)
    S, B = 3, 5
    m = WHVISquarePow2Matrix(D, bias=True, covariance=covariance).to(dev())
    g = _gen(D)
    eps = _randn((S, D), g)
    x = _randn((S, B, D), g, torch.bfloat16).requires_grad_()
    dy = _randn((S, B, D), g, torch.bfloat16)
    m.inject_eps(eps)
    y = m(x)
    assert y.dtype == torch.bfloat16 and y.shape == (S, B, D)
    y.backward(dy)
    assert x.grad.dtype == torch.bfloat16
    assert all(p.grad.dtype == torch.float32 for p in m.parameters())
    with torch.no_grad():
        gs = m._g(eps)
        _eq(y.detach(), F.layer_forward_bf16(x.detach(), gs, m.s1, m.s2, m.bias.reshape(-1)), "y")
        dx, dg, ds1, ds2, db = F.layer_backward_raw(x.detach(), dy, gs, m.s1, m.s2, want_dbias=True)
    _eq(x.grad, dx, "dx")
    _eq(m.s1.grad, ds1, "ds1")
    _eq(m.s2.grad, ds2, "ds2")
    _eq(m.bias.grad, db.reshape(1, D), "dbias")
    mu = m.g_mu.detach().requires_grad_()
    if covariance == "diag":
        rho = m.g_rho.detach().requires_grad_()
        F.reparam(mu, rho, eps).backward(dg)
        _eq(m.g_rho.grad, rho.grad, "drho")
    else:
        L = m.g_L.detach().requires_grad_()
        F.reparam_dense(mu, L, eps).backward(dg)
        _eq(m.g_L.grad, L.grad, "dL")
    _eq(m.g_mu.grad, mu.grad, "dmu")


def _regression(D, bias, seed):
    from whvi_b200.layers import WHVILinear
    from whvi_b200.networks import WHVIRegression
    torch.manual_seed(seed)
    return WHVIRegression([WHVILinear(D, D, bias=bias), torch.nn.ReLU(), WHVILinear(D, D, bias=bias), torch.nn.ReLU(),
                           WHVILinear(D, D, bias=bias)], sigma=0.7, train_samples=3).to(dev())


# bf16 vs fp32 network, max|diff| / max|fp32| per quantity.  Loose: every layer boundary rounds the activations to 8 significant
# bits.  The bias gradients are sums of dy over only S * B = 18 rows, where cancellation magnifies that rounding (measured on a
# B200: up to 0.27 for the biases, up to 0.07 for everything else).
FP32_VS_BF16_TOL, FP32_VS_BF16_TOL_BIAS = 0.1, 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1024, 4096])
def test_network_bf16_equals_explicit_kernel_composition(D):
    """Three square layers with ReLUs (both fused), fused loss layer, deferred loss scale: the network's loss and every
    parameter gradient equal, bit for bit, the fp32 kernels composed by hand with bf16 rounding at each layer boundary."""
    from whvi_b200 import functional as F
    B, S, n = 6, 3, 100
    net = _regression(D, True, D)
    g = _gen(D + 1)
    X = _randn((B, D), g)
    Y = _randn((B, D), g)
    eps = [_randn((S, D), g) for _ in range(3)]
    blocks = [layer.weight_submodule for layer in net._whvi_layers()]

    def run(x):
        net.zero_grad(set_to_none=True)
        for b, e in zip(blocks, eps):
            b.inject_eps(e)
        loss = net.loss(x, Y, n=n)
        loss.backward()
        return loss.detach(), {k: p.grad.clone() for k, p in net.named_parameters()}

    loss, grads = run(X.to(torch.bfloat16))

    # explicit composition: the fp32 kernels on widened inputs, every activation and dx rounded to bf16 at the layer boundary
    bf = torch.bfloat16
    with torch.no_grad():
        gs = [F.reparam(b.g_mu, b.g_rho, e) for b, e in zip(blocks, eps)]
        bias = [b.bias.reshape(-1) for b in blocks]
        h0 = X.to(bf)
        h1 = F.layer_forward_raw(h0.float(), gs[0], blocks[0].s1, blocks[0].s2, bias[0], relu_out=True).to(bf)
        h2 = F.layer_forward_raw(h1.float(), gs[1], blocks[1].s1, blocks[1].s2, bias[1], relu_out=True).to(bf)
        sq, dx3, dg3, ds1_3, ds2_3, db3 = F.layer_loss_raw(h2.float(), gs[2], blocks[2].s1, blocks[2].s2, bias[2], Y,
                                                           relu_in=True)
        assert dx3.dtype == torch.float32
        dx3 = dx3.to(bf)
    sq_leaf = sq.clone().requires_grad_()
    lik = type(net.likelihood)(0.7).to(dev())
    mnll = lik.mnll_from_sq_error(sq_leaf, m=B, n_out=D, n_mc=S, n=n)
    kls = [F.kl_gaussian(b.g_mu, b.g_rho, b.lambda_, b.kl_mode) for b in blocks]
    ref_loss = mnll + sum(kls)
    _eq(loss, ref_loss.detach(), "loss")
    mnll.backward()
    c = (2.0 * sq_leaf.grad).to(torch.float32)
    _eq(grads["likelihood.sigma"], lik.sigma.grad, "dsigma")
    with torch.no_grad():
        dx2, dg2, ds1_2, ds2_2, db2 = F.layer_backward_raw(h1.float(), dx3.float(), gs[1], blocks[1].s1, blocks[1].s2,
                                                           want_dbias=True, relu_in=True, dy_scale=c.reshape(1))
        assert dx2.dtype == torch.float32
        dx2 = dx2.to(bf)
        _, dg1, ds1_1, ds2_1, db1 = F.layer_backward_raw(h0.float(), dx2.float(), gs[0], blocks[0].s1, blocks[0].s2,
                                                         want_dx=False, want_dbias=True)
    per_layer = [(dg1, ds1_1, ds2_1, db1), (dg2, ds1_2, ds2_2, db2), (dg3 * c, ds1_3 * c, ds2_3 * c, db3 * c)]
    for i, (b, e, (dg, ds1, ds2, db)) in enumerate(zip(blocks, eps, per_layer)):
        p = f"sequential.{2 * i}.weight_submodule."
        _eq(grads[p + "s1"], ds1, f"layer {i} ds1")
        _eq(grads[p + "s2"], ds2, f"layer {i} ds2")
        _eq(grads[p + "bias"], db.reshape(1, D), f"layer {i} dbias")
        mu, rho = b.g_mu.detach().requires_grad_(), b.g_rho.detach().requires_grad_()
        F.reparam(mu, rho, e).backward(dg)
        kmu, krho = b.g_mu.detach().requires_grad_(), b.g_rho.detach().requires_grad_()
        F.kl_gaussian(kmu, krho, b.lambda_, b.kl_mode).backward()
        _eq(grads[p + "g_mu"], mu.grad + kmu.grad, f"layer {i} dmu")
        _eq(grads[p + "g_rho"], rho.grad + krho.grad, f"layer {i} drho")

    # the same network in fp32: reported, and within a loose tolerance
    loss32, grads32 = run(X)
    errs = {"loss": abs(loss.item() - loss32.item()) / abs(loss32.item())}
    for k in grads:
        d = grads32[k].abs().max().item()
        errs[k] = (grads[k] - grads32[k]).abs().max().item() / (d if d > 0 else 1.0)
    print(f"D={D} bf16 vs fp32 network, max|diff|/max|fp32|: " + ", ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    for k, v in errs.items():
        assert v < (FP32_VS_BF16_TOL_BIAS if k.endswith("bias") else FP32_VS_BF16_TOL), (k, errs)


@pytest.mark.gpu
def test_network_bf16_without_fused_loss_and_predictive_sums():
    """loss() without grad (bf16 forward + closed-form MNLL) and eval paths accept bf16 inputs."""
    D, B, S = 256, 4, 3
    net = _regression(D, False, 7)
    g = _gen(11)
    X, Y = _randn((B, D), g), _randn((B, D), g)
    blocks = [layer.weight_submodule for layer in net._whvi_layers()]
    eps = [_randn((S, D), g) for _ in range(3)]
    for b, e in zip(blocks, eps):
        b.inject_eps(e)
    with torch.no_grad():
        net.loss(X.to(torch.bfloat16), Y, n=10)
        mnll = net.current_mnll
    for b, e in zip(blocks, eps):
        b.inject_eps(e)
    with torch.no_grad():
        pred = net(X.to(torch.bfloat16))           # (B, D, S), bf16
    assert pred.dtype == torch.bfloat16
    ref = net.likelihood.mnll_from_sq_error((pred.float() - Y.unsqueeze(-1)).square().sum(), m=B, n_out=D, n_mc=S, n=10)
    torch.testing.assert_close(mnll, ref, rtol=1e-5, atol=0)
    net.eval_samples = S
    for b, e in zip(blocks, eps):
        b.inject_eps(e)
    sum_y, sum_y2, n_s = net.predictive_sums(X.to(torch.bfloat16))
    assert n_s == S and sum_y.dtype == torch.float32
    ref_y = pred.float().sum(-1)   # bf16 predictions; the moments are taken on the last layer's fp32 output
    assert (sum_y - ref_y).abs().max() <= 1e-2 * ref_y.abs().max()
    rmse, mnll = net.eval_model(X.to(torch.bfloat16), Y)
    assert rmse == rmse and mnll == mnll


@pytest.mark.gpu
def test_cuda_graph_bf16_step_matches_eager():
    """A graph-captured training step on bf16 minibatches equals the eager step bit for bit.  The posterior noise is
    switched off (softplus(-30) ~ 1e-13 vanishes next to O(1) means), so both runs see the same weights."""
    import copy
    from whvi_b200.graphs import GraphedTrainStep
    D, B, n = 1024, 8, 64
    eager = _regression(D, True, 3)
    with torch.no_grad():
        for name, p in eager.named_parameters():
            if name.endswith("g_mu"):
                p.normal_()
            if name.endswith("g_rho"):
                p.fill_(-30.0)
    graphed = copy.deepcopy(eager)
    g = _gen(3)
    xs = [_randn((B, D), g, torch.bfloat16) for _ in range(3)]
    ys = [_randn((B, D), g) for _ in range(3)]
    opt_e = torch.optim.Adam(eager.parameters(), lr=torch.tensor(1e-3, device=dev()), capturable=True)
    opt_g = torch.optim.Adam(graphed.parameters(), lr=torch.tensor(1e-3, device=dev()), capturable=True)
    step = GraphedTrainStep(graphed, opt_g, xs[0], ys[0], n=n)
    assert step.x.dtype == torch.bfloat16
    for it, (x, y) in enumerate(zip(xs, ys)):
        loss_e = eager.loss(x, y, n=n)
        loss_e.backward()
        opt_e.step()
        opt_e.zero_grad(set_to_none=True)
        loss_g = step(x, y)
        _eq(loss_g.detach(), loss_e.detach(), f"loss, step {it}")
        for (k, pe), pg in zip(eager.named_parameters(), graphed.parameters()):
            _eq(pg.detach(), pe.detach(), f"{k}, step {it}")
