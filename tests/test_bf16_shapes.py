"""bf16 activations for the Stacked and Column layers: ``whvi_stacked_{fwd,bwd}[_g]_bf16``, ``whvi_column_{fwd,bwd}[_g]_bf16``,
``whvi_pad_rows_bf16`` and everything above them.

Definition checked throughout: a bf16 call is the fp32 call on the widened inputs.  Parameter gradients (and dg) are bit-identical
to the fp32 call's for float(x), float(dy); every bf16 output (y, dx) is the fp32 output rounded once -- for a Stacked layer with
several blocks too, whose per-block dx are summed in fp32 before the rounding.  The transposed Column layer's output and its
gradient stay fp32.  The CPU tests check argument validation only; the GPU tests check the definition with ``torch.equal``."""
import pytest
import torch

E_NULL, E_SHAPE, E_ALIGN, E_MODE, E_WORKSPACE = -1, -2, -3, -4, -5
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference


def _args(base, **kw):
    a = dict(base)
    a.update(kw)
    return tuple(a.values())


PAD = dict(inp=A, out=A, rows=6, n_in=13, D=16, stream=None)
SFWD = dict(x=A, xs=0, mu=A, rho=A, s1=A, s2=A, pstride=16, eps=A, bias=None, g=A, yb=A, y=A, S=2, B=3, D=16, G=8, n_out=128,
            flags=0, stream=None)
SFWD_G = dict(x=A, xs=0, g=A, s1=A, s2=A, pstride=16, bias=None, yb=A, y=A, S=2, B=3, D=16, G=8, n_out=128, flags=0, stream=None)
SBWD = dict(x=A, xs=0, dy=A, g=A, rho=A, s1=A, s2=A, pstride=16, eps=A, dx=A, n_in=13, dmu=A, drho=A, ds1=A, ds2=A, dbias=None, ws=A,
            ws_bytes=1 << 30, S=2, B=4, D=16, G=8, n_out=128, flags=0, stream=None)
SBWD_G = dict(x=A, xs=0, dy=A, g=A, s1=A, s2=A, pstride=16, dx=A, n_in=13, dg=A, ds1=A, ds2=A, dbias=None, ws=A, ws_bytes=1 << 30,
              S=2, B=4, D=16, G=8, n_out=128, flags=0, stream=None)
CFWD = dict(x=A, xs=0, mu=A, rho=A, s1=A, s2=A, eps=A, bias=None, g=A, hg=A, y=A, S=2, B=3, D=128, n=100, transposed=1, flags=0,
            stream=None)
CFWD_G = dict(x=A, xs=0, g=A, s1=A, s2=A, bias=None, hg=A, y=A, S=2, B=3, D=128, n=100, transposed=1, flags=0, stream=None)
CBWD = dict(x=A, xs=0, dy=A, hg=A, rho=A, s1=A, s2=A, eps=A, dx=A, dmu=A, drho=A, ds1=A, ds2=A, dbias=None, ws=A, ws_bytes=1 << 30,
            S=2, B=3, D=128, n=100, transposed=1, flags=0, stream=None)
CBWD_G = dict(x=A, xs=0, dy=A, hg=A, s1=A, s2=A, dx=A, dg=A, ds1=A, ds2=A, dbias=None, ws=A, ws_bytes=1 << 30, S=2, B=3, D=128, n=100,
              transposed=1, flags=0, stream=None)

CASES = {
    "whvi_pad_rows_bf16": [
        (_args(PAD, D=8), E_SHAPE, "pad_rows_bf16"),
        (_args(PAD, inp=None), E_NULL, "null pointer"),
        (_args(PAD, out=A + 8), E_ALIGN, "16-byte"),
        (_args(PAD, inp=A + 1), E_ALIGN, "2-byte"),
    ],
    "whvi_stacked_fwd_bf16": [
        (_args(SFWD, D=2), E_SHAPE, "outside"),
        (_args(SFWD, G=2), E_SHAPE, "do not match"),
        (_args(SFWD, pstride=6), E_SHAPE, "param_stride"),
        (_args(SFWD, xs=5), E_SHAPE, "x_sample_stride"),
        (_args(SFWD, flags=2), E_MODE, "unknown flags"),
        (_args(SFWD, eps=None), E_NULL, "null pointer"),
        (_args(SFWD, yb=None), E_NULL, "null pointer"),
        (_args(SFWD, g=A + 4), E_ALIGN, "16-byte"),
        (_args(SFWD, x=A + 4), E_ALIGN, "8-byte"),
        (_args(SFWD, yb=A + 2), E_ALIGN, "8-byte"),
        (_args(SFWD, y=A + 1), E_ALIGN, "2-byte"),
    ],
    "whvi_stacked_fwd_g_bf16": [
        (_args(SFWD_G, n_out=129), E_SHAPE, "do not match"),
        (_args(SFWD_G, flags=4), E_MODE, "unknown flags"),
        (_args(SFWD_G, g=None), E_NULL, "null pointer"),
        (_args(SFWD_G, s1=A + 4), E_ALIGN, "16-byte"),
        (_args(SFWD_G, x=A + 2), E_ALIGN, "8-byte"),
    ],
    "whvi_stacked_bwd_bf16": [
        (_args(SBWD, D=16384), E_SHAPE, "outside"),
        (_args(SBWD, flags=2), E_MODE, "unknown flags"),
        (_args(SBWD, n_in=17), E_SHAPE, "n_in"),
        (_args(SBWD, drho=None), E_NULL, "null output"),
        (_args(SBWD, eps=None), E_NULL, "null pointer"),
        (_args(SBWD, x=A + 8), E_ALIGN, "16-byte"),              # the padded x arrives by bulk copy
        (_args(SBWD, D=4, G=32, pstride=4, B=5, n_in=3), E_SHAPE, "multiple of 8"),
        (_args(SBWD, dy=A + 1), E_ALIGN, "2-byte"),
        (_args(SBWD, dx=A + 1), E_ALIGN, "2-byte"),
        (_args(SBWD, ws_bytes=64), E_WORKSPACE, "workspace"),
    ],
    "whvi_stacked_bwd_g_bf16": [
        (_args(SBWD_G, G=9), E_SHAPE, "do not match"),
        (_args(SBWD_G, dg=None), E_NULL, "null output"),
        (_args(SBWD_G, dy=None), E_NULL, "null pointer"),
        (_args(SBWD_G, dg=A + 4), E_ALIGN, "16-byte"),
        (_args(SBWD_G, B=3, D=4, G=32, pstride=4, n_in=3), E_SHAPE, "multiple of 8"),
        (_args(SBWD_G, ws=A + 4), E_ALIGN, "16-byte"),
        (_args(SBWD_G, ws_bytes=64), E_WORKSPACE, "workspace"),
    ],
    "whvi_column_fwd_bf16": [
        (_args(CFWD, n=64), E_SHAPE, "next_pow2"),
        (_args(CFWD, xs=7), E_SHAPE, "x_sample_stride"),
        (_args(CFWD, flags=1), E_MODE, "RELU_OUT"),
        (_args(CFWD, mu=None), E_NULL, "null pointer"),
        (_args(CFWD, hg=A + 4), E_ALIGN, "16-byte"),
        (_args(CFWD, x=A + 1), E_ALIGN, "2-byte"),
        (_args(CFWD, transposed=0, y=A + 1), E_ALIGN, "2-byte"),
    ],
    "whvi_column_fwd_g_bf16": [
        (_args(CFWD_G, D=96), E_SHAPE, "next_pow2"),
        (_args(CFWD_G, flags=2), E_MODE, "unknown flags"),
        (_args(CFWD_G, g=None), E_NULL, "null pointer"),
        (_args(CFWD_G, x=A + 1), E_ALIGN, "2-byte"),
    ],
    "whvi_column_bwd_bf16": [
        (_args(CBWD, n=300), E_SHAPE, "next_pow2"),
        (_args(CBWD, transposed=0, flags=1), E_MODE, "RELU_IN"),
        (_args(CBWD, dmu=None), E_NULL, "null output"),
        (_args(CBWD, rho=None), E_NULL, "null pointer"),
        (_args(CBWD, ws=A + 4), E_ALIGN, "16-byte"),
        (_args(CBWD, dx=A + 1), E_ALIGN, "2-byte"),
        (_args(CBWD, transposed=0, dy=A + 1), E_ALIGN, "2-byte"),
        (_args(CBWD, ws_bytes=64), E_WORKSPACE, "workspace"),
    ],
    "whvi_column_bwd_g_bf16": [
        (_args(CBWD_G, flags=2), E_MODE, "unknown flags"),
        (_args(CBWD_G, dg=None), E_NULL, "null output"),
        (_args(CBWD_G, dg=A + 4), E_ALIGN, "dg"),
        (_args(CBWD_G, x=A + 1), E_ALIGN, "2-byte"),
        (_args(CBWD_G, ws_bytes=64), E_WORKSPACE, "workspace"),
    ],
}


def test_bf16_shape_entry_points_validate_before_any_cuda_call():
    from whvi_b200 import _lib
    L = _lib.lib()
    for name, cases in CASES.items():
        for args, code, msg in cases:
            assert getattr(L, name)(*args) == code, (name, args, L.whvi_last_error())
            assert msg in L.whvi_last_error().decode(), (name, args, L.whvi_last_error())
    # an empty batch is a no-op forward (nothing is dereferenced)
    assert L.whvi_stacked_fwd_bf16(*_args(SFWD, B=0)) == 0
    assert L.whvi_column_fwd_bf16(*_args(CFWD, S=0)) == 0


def test_bf16_shape_entry_points_shim_matches_ctypes():
    from whvi_b200 import _lib
    L = _lib.lib()
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    for name, cases in CASES.items():
        fast, raw = getattr(L, name), getattr(L._cdll, name)
        assert not hasattr(fast, "argtypes"), name
        for args, _, _ in cases:
            rc_fast, msg_fast = fast(*args), L.whvi_last_error()
            rc_raw, msg_raw = raw(*args), L.whvi_last_error()
            assert rc_fast == rc_raw < 0 and msg_fast == msg_raw and msg_fast, (name, args)


def test_every_bf16_shape_entry_point_is_counted():
    from whvi_b200 import functional as F
    for name in CASES:
        assert F._LAUNCHES_PER_CALL[name] == F._LAUNCHES_PER_CALL[name.replace("_bf16", "_f32")], name


def test_bf16_on_cpu_names_bf16():
    """Stacked and Column modules take bf16 on CUDA only; on the CPU the error says so (nothing upcasts)."""
    from whvi_b200.weights import WHVIColumnMatrix, WHVIStackedMatrix
    for module, x in ((WHVIStackedMatrix(13, 128), torch.zeros(3, 13, dtype=torch.bfloat16)),
                      (WHVIColumnMatrix(100, transposed=True), torch.zeros(3, 100, dtype=torch.bfloat16)),
                      (WHVIColumnMatrix(100), torch.zeros(3, 1, dtype=torch.bfloat16))):
        with pytest.raises(RuntimeError, match="bf16 activations run on CUDA only"):
            module(x)


# ------------------------------------------------------------------------------------------------------------------- GPU
def dev():
    return torch.device("cuda:0")


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _randn(shape, g, dtype=torch.float32):
    return torch.randn(shape, generator=g, device=dev()).to(dtype)


def _eq(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    assert torch.equal(a, b), f"{what}: max |diff| {(a.float() - b.float()).abs().max().item()}"


bf = torch.bfloat16


def _grads(out, inputs, dout):
    return torch.autograd.grad(out, inputs, dout, allow_unused=True)


# (n_in, n_out, S, B): D = next_pow2(n_in), G = ceil(n_out / D).  n_in % 4 != 0 pads the input rows on the vector-less path; B odd at
# D = 4 takes the zero-row padding of the backward; n_out not a multiple of D drops the padded columns; D >= 2048 runs the
# tensor-memory backward.
STACKED_SHAPES = [(3, 16, 3, 5), (13, 128, 2, 7), (16, 40, 2, 6), (100, 300, 2, 6), (128, 512, 3, 9), (1000, 2500, 2, 3),
                  (2048, 4096, 2, 3), (4000, 5000, 2, 2), (8192, 8292, 1, 2)]
STACKED_FLAGS = [(True, False, False), (False, True, True)]   # (bias, relu_out, relu_in)


@pytest.mark.gpu
@pytest.mark.parametrize("n_in,n_out,S,B", STACKED_SHAPES)
@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("form", ["diag", "g"])
def test_stacked_bf16_is_fp32_on_widened_inputs(n_in, n_out, S, B, shared, form):
    from whvi_b200 import functional as F
    D = 1 << max(2, (n_in - 1).bit_length())
    G = -(-n_out // D)
    r = _gen(n_in * 7 + n_out + B)
    s1 = [_randn(D, r).requires_grad_() for _ in range(G)]
    s2 = [_randn(D, r).requires_grad_() for _ in range(G)]
    mu = [_randn(D, r).requires_grad_() for _ in range(G)]
    rho = [(_randn(D, r) - 2).requires_grad_() for _ in range(G)]
    eps = _randn((G, S, D), r)
    g = _randn((G, S, D), r).requires_grad_()
    x = _randn((B, n_in) if shared else (S, B, n_in), r, bf)
    dy = _randn((S, B, n_out), r, bf)
    for has_bias, relu_out, relu_in in STACKED_FLAGS:
        bias = _randn((1, G * D), r).requires_grad_() if has_bias else None
        tag = f"n_in={n_in} n_out={n_out} S={S} B={B} shared={shared} form={form} bias={has_bias} relu={relu_out}"
        outs = []
        for xin, dyin in ((x, dy), (x.float(), dy.float())):
            xin = xin.clone().requires_grad_()
            if form == "diag":
                y = F.whvi_stacked(xin, eps, bias, n_out, s1, s2, mu, rho, relu_out=relu_out, relu_in=relu_in)
                params = s1 + s2 + mu + rho
            else:
                y = F.whvi_stacked_g(xin, g, bias, n_out, s1, s2, relu_out=relu_out, relu_in=relu_in)
                params = s1 + s2 + [g]
            params = params + ([bias] if has_bias else [])
            outs.append((y, _grads(y, [xin] + params, dyin)))
        (y16, gr16), (y32, gr32) = outs
        _eq(y16, y32.to(bf), f"y {tag}")
        if shared:   # dx of a shared input is the bf16 per-sample dx summed over the samples in torch
            assert gr16[0].dtype == bf and gr16[0].shape == (B, n_in)
        else:
            _eq(gr16[0], gr32[0].to(bf), f"dx {tag}")
        for i, (a, b) in enumerate(zip(gr16[1:], gr32[1:])):
            _eq(a, b, f"param grad {i} {tag}")


# (n, S, B) with D = next_pow2(n)
COLUMN_SHAPES = [(3, 3, 5), (100, 2, 7), (128, 2, 33), (1000, 3, 4), (4097, 2, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,S,B", COLUMN_SHAPES)
@pytest.mark.parametrize("transposed", [True, False])
@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("form", ["diag", "g"])
def test_column_bf16_is_fp32_on_widened_inputs(n, S, B, transposed, shared, form):
    from whvi_b200 import functional as F
    D = 1 << max(0, (n - 1).bit_length())
    r = _gen(n * 3 + B + transposed)
    s1, s2, mu = _randn(D, r).requires_grad_(), _randn(D, r).requires_grad_(), _randn(D, r).requires_grad_()
    rho = (_randn(D, r) - 2).requires_grad_()
    eps = _randn((S, D), r)
    g = _randn((S, D), r).requires_grad_()
    width = n if transposed else 1
    x = _randn((B, width) if shared else (S, B, width), r, bf)
    dy = _randn((S, B, 1 if transposed else n), r, torch.float32 if transposed else bf)   # the transposed form's dy is fp32
    for has_bias, relu in ((True, False), (False, True)):
        bias = _randn((1, 1 if transposed else n), r).requires_grad_() if has_bias else None
        relu_out, relu_in = (False, relu) if transposed else (relu, False)
        tag = f"n={n} S={S} B={B} transposed={transposed} shared={shared} form={form} bias={has_bias} relu={relu}"
        outs = []
        for xin, dyin in ((x, dy), (x.float(), dy.float())):
            xin = xin.clone().requires_grad_()
            if form == "diag":
                y = F.whvi_column(xin, eps, mu, rho, s1, s2, bias, n, transposed, relu_out, relu_in)
                params = [mu, rho, s1, s2]
            else:
                y = F.whvi_column_g(xin, g, s1, s2, bias, n, transposed, relu_out, relu_in)
                params = [g, s1, s2]
            params = params + ([bias] if has_bias else [])
            outs.append((y, _grads(y, [xin] + params, dyin)))
        (y16, gr16), (y32, gr32) = outs
        _eq(y16, y32 if transposed else y32.to(bf), f"y {tag}")
        if shared:
            assert gr16[0].dtype == bf and gr16[0].shape == (B, width)
        else:
            _eq(gr16[0], gr32[0].to(bf), f"dx {tag}")
        for i, (a, b) in enumerate(zip(gr16[1:], gr32[1:])):
            _eq(a, b, f"param grad {i} {tag}")


@pytest.mark.gpu
@pytest.mark.parametrize("covariance", ["diag", "dense"])
@pytest.mark.parametrize("kind", ["stacked", "column", "column_t"])
def test_modules_autograd_bf16(kind, covariance):
    """Module forward + autograd with bf16 input against the same module on the widened input: output rounded once (fp32 for the
    transposed Column layer), dx rounded once, every parameter gradient fp32 and bit-identical."""
    from whvi_b200.weights import WHVIColumnMatrix, WHVIStackedMatrix
    torch.manual_seed(5)
    S, B = 3, 6
    if kind == "stacked":
        m, n_in, n_out = WHVIStackedMatrix(100, 300, bias=True, covariance=covariance), 100, 300
        blocks = list(m.weight_matrices)
    else:
        t = kind == "column_t"
        m = WHVIColumnMatrix(100, bias=True, transposed=t, covariance=covariance)
        n_in, n_out = (100, 1) if t else (1, 100)
        blocks = [m.weight_submodule]
    m = m.to(dev())
    r = _gen(9)
    eps = [_randn((S, b.D), r) for b in blocks]
    x = _randn((S, B, n_in), r, bf)
    dy = _randn((S, B, n_out), r, torch.float32 if kind == "column_t" else bf)
    res = []
    for xin, dyin in ((x, dy), (x.float(), dy.float())):
        for b, e in zip(blocks, eps):
            b.inject_eps(e)
        m.zero_grad(set_to_none=True)
        xin = xin.clone().requires_grad_()
        y = m(xin)
        y.backward(dyin)
        res.append((y.detach(), xin.grad, {k: p.grad.clone() for k, p in m.named_parameters()}))
    (y16, dx16, g16), (y32, dx32, g32) = res
    _eq(y16, y32 if kind == "column_t" else y32.to(bf), "y")
    _eq(dx16, dx32.to(bf), "dx")
    assert set(g16) == set(g32)
    for k in g16:
        _eq(g16[k], g32[k], k)


@pytest.mark.gpu
def test_unsupported_bf16_paths_raise_on_gpu():
    """No kernel, no bf16: the reference semantics, the block-by-block Stacked path and the unfused Column op chain raise."""
    from whvi_b200.weights import WHVIColumnMatrix, WHVIStackedMatrix
    x = torch.zeros(3, 13, dtype=bf, device=dev())
    with pytest.raises(RuntimeError, match="bf16"):
        WHVIStackedMatrix(13, 128, semantics="reference").to(dev())(x)
    m = WHVIStackedMatrix(13, 128).to(dev())
    m.one_launch = False
    with pytest.raises(RuntimeError, match="bf16"):
        m(x)
    with pytest.raises(RuntimeError, match="bf16"):
        WHVIStackedMatrix(10000, 10000 + 1).to(dev())(torch.zeros(2, 10000, dtype=bf, device=dev()))   # D_in = 16384
    c = WHVIColumnMatrix(13, transposed=True).to(dev())
    c.one_launch = False
    with pytest.raises(RuntimeError, match="bf16"):
        c(x)
    with pytest.raises(RuntimeError, match="bf16"):
        WHVIColumnMatrix(13, transposed=True, semantics="reference").to(dev())(x)


# ---------------------------------------------------------------------------------------------------------------- networks
class _RoundBF16(torch.autograd.Function):
    """A layer boundary of the bf16 network: the activation and the gradient that crosses it back are rounded to bf16 (and
    widened again for the next fp32 call)."""

    @staticmethod
    def forward(ctx, h):
        return h.to(bf).float()

    @staticmethod
    def backward(ctx, d):
        return d.to(bf).float()


def _net(widths, seed, covariance="diag", samples=3):
    from whvi_b200.layers import WHVILinear
    from whvi_b200.networks import WHVIRegression
    torch.manual_seed(seed)
    mods = []
    for i, (a, b) in enumerate(zip(widths[:-1], widths[1:])):
        if i:
            mods.append(torch.nn.ReLU())
        mods.append(WHVILinear(a, b, bias=True, covariance=covariance))
    return WHVIRegression(mods, sigma=0.7, train_samples=samples).to(dev())


def _composed_loss(net, X, Y, n):
    """The network's loss from the fp32 layer calls, with the activations and their gradients rounded to bf16 at every layer
    boundary (the transposed Column layer's output is not an activation: it stays fp32), the ReLUs fused as the network does."""
    layers = net._whvi_layers()
    S = net.train_samples
    for layer in layers:
        layer.mc_samples = S
    try:
        h = _RoundBF16.apply(X)
        for i, layer in enumerate(layers):
            w = layer.weight_submodule
            last = i == len(layers) - 1
            h = w.forward(h, relu_out=not last, relu_in=i > 0)
            if not (last and getattr(w, "transposed", False)):
                h = _RoundBF16.apply(h)
    finally:
        for layer in layers:
            layer.mc_samples = None
    pred = h.reshape(S, X.size(0), -1).permute(1, 2, 0)
    return net.likelihood.mnll_batch_estimate(Y, pred, n) + net.kl


NETS = {"c1": [3, 16, 1], "c3": [13, 128, 128, 1], "mid_stacked": [13, 128, 512, 1]}
# bf16 vs fp32 network, max|diff| / max|fp32| per quantity: loose, every layer boundary rounds the activations to 8 significant bits
FP32_VS_BF16_TOL, FP32_VS_BF16_TOL_BIAS = 0.1, 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("net_name,covariance", [("c1", "diag"), ("c3", "diag"), ("mid_stacked", "diag"), ("c3", "dense")])
def test_network_bf16_equals_explicit_composition(net_name, covariance):
    widths = NETS[net_name]
    B, n = 7 if net_name == "c1" else 10, 100   # config 1's odd minibatch: D = 4 with an odd B
    net = _net(widths, 17, covariance)
    r = _gen(23)
    X, Y = _randn((B, widths[0]), r), _randn((B, 1), r)
    blocks = [b for layer in net._whvi_layers() for b in layer.square_blocks()]
    eps = [_randn((net.train_samples, b.D), r) for b in blocks]

    def run(loss_fn):
        net.zero_grad(set_to_none=True)
        for b, e in zip(blocks, eps):
            b.inject_eps(e)
        loss = loss_fn()
        loss.backward()
        return loss.detach(), {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}

    loss16, g16 = run(lambda: net.loss(X.to(bf), Y, n=n))
    ref, gref = run(lambda: _composed_loss(net, X, Y, n))
    _eq(loss16, ref, "loss")
    assert set(g16) == set(gref) and len(g16) == len(list(net.parameters()))
    for k in g16:
        _eq(g16[k], gref[k], k)
    assert all(g.dtype == torch.float32 for g in g16.values())

    loss32, g32 = run(lambda: net.loss(X, Y, n=n))
    errs = {"loss": abs(loss16.item() - loss32.item()) / abs(loss32.item())}
    for k in g16:
        d = g32[k].abs().max().item()
        errs[k] = (g16[k] - g32[k]).abs().max().item() / (d if d > 0 else 1.0)
    print(f"{net_name}/{covariance} bf16 vs fp32 network, max|diff|/max|fp32|: " + ", ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    for k, v in errs.items():
        assert v < (FP32_VS_BF16_TOL_BIAS if k.endswith("bias") else FP32_VS_BF16_TOL), (k, errs)


@pytest.mark.gpu
def test_network_bf16_launches_match_fp32():
    """A bf16 config-3 training step issues exactly the fp32 step's kernel launches."""
    from whvi_b200 import functional as F
    net = _net(NETS["c3"], 3)
    r = _gen(4)
    X, Y = _randn((64, 13), r), _randn((64, 1), r)
    counts = []
    for x in (X, X.to(bf)):
        F.LAUNCH_COUNTS.clear()
        net.loss(x, Y, n=100).backward()
        counts.append(sum(F.LAUNCH_COUNTS.values()))
    assert counts[0] == counts[1], counts


@pytest.mark.gpu
def test_cuda_graph_bf16_config3_step_matches_eager():
    """A graph-captured config-3 training step on bf16 minibatches equals the eager step bit for bit.  The posterior noise is
    switched off (softplus(-30) ~ 1e-13 vanishes next to O(1) means), so both runs see the same weights."""
    import copy
    from whvi_b200.graphs import GraphedTrainStep
    B, n = 64, 500
    eager = _net(NETS["c3"], 5)
    with torch.no_grad():
        for name, p in eager.named_parameters():
            if name.endswith("g_mu"):
                p.normal_()
            if name.endswith("g_rho"):
                p.fill_(-30.0)
    graphed = copy.deepcopy(eager)
    r = _gen(6)
    xs = [_randn((B, 13), r, bf) for _ in range(3)]
    ys = [_randn((B, 1), r) for _ in range(3)]
    opt_e = torch.optim.Adam(eager.parameters(), lr=torch.tensor(1e-3, device=dev()), capturable=True)
    opt_g = torch.optim.Adam(graphed.parameters(), lr=torch.tensor(1e-3, device=dev()), capturable=True)
    step = GraphedTrainStep(graphed, opt_g, xs[0], ys[0], n=n)
    assert step.x.dtype == bf
    for it, (x, y) in enumerate(zip(xs, ys)):
        loss_e = eager.loss(x, y, n=n)
        loss_e.backward()
        opt_e.step()
        opt_e.zero_grad(set_to_none=True)
        loss_g = step(x, y)
        _eq(loss_g.detach(), loss_e.detach(), f"loss, step {it}")
        for (k, pe), pg in zip(eager.named_parameters(), graphed.parameters()):
            _eq(pg.detach(), pe.detach(), f"{k}, step {it}")


@pytest.mark.gpu
def test_train_model_cuda_graph_and_flat_adam_bf16():
    """train_model(cuda_graph=True) with FlatAdam on bf16 minibatches of a config-3-shaped model runs and moves the parameters."""
    from whvi_b200.optim import FlatAdam, FlatParams
    net = _net(NETS["c3"], 8)
    r = _gen(8)
    data = torch.utils.data.TensorDataset(_randn((128, 13), r, bf), _randn((128, 1), r))
    loader = torch.utils.data.DataLoader(data, batch_size=64)
    opt = FlatAdam(FlatParams(net.parameters()), lr=torch.tensor(1e-3, device=dev()))
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda e: 1.0)
    before = [p.detach().clone() for p in net.parameters()]
    net.train_model(loader, opt, sched, epochs1=2, epochs2=1, cuda_graph=True)
    moved = [not torch.equal(a, p.detach()) for a, p in zip(before, net.parameters())]
    assert all(moved[:-1]) and float(net.current_mnll) == float(net.current_mnll)


@pytest.mark.gpu
@pytest.mark.parametrize("net_name", ["c1", "c3"])
def test_eval_and_forward_accept_bf16_for_column_final_networks(net_name):
    widths = NETS[net_name]
    net = _net(widths, 31)
    r = _gen(31)
    X, Y = _randn((9, widths[0]), r), _randn((9, 1), r)
    net.eval_samples = 4
    blocks = [b for layer in net._whvi_layers() for b in layer.square_blocks()]
    eps = [_randn((4, b.D), r) for b in blocks]
    for b, e in zip(blocks, eps):
        b.inject_eps(e)
    net.eval()
    with torch.no_grad():
        pred = net(X.to(bf))
    assert pred.shape == (9, 1, 4) and pred.dtype == torch.float32   # the transposed Column layer's output stays fp32
    assert net.predictive_sums(X.to(bf)) is None
    for b, e in zip(blocks, eps):
        b.inject_eps(e)
    rmse, mnll = net.eval_model(X.to(bf), Y)
    ref = torch.sqrt(((pred.mean(dim=2) - Y) ** 2).mean()).item()
    assert rmse == pytest.approx(ref, rel=1e-5) and mnll == mnll
