"""Classification: the categorical (softmax) likelihood from the sm_100a kernels (``csrc/categorical.cu``) up to
``WHVIClassification``.

CPU: argument validation of the new entry points (shim and ctypes alike), their bindings and launch counts, the fp64 numpy
restatement against torch fp64, the Python front end's input checks and the network's state_dict.
GPU: the kernels against the fp64 restatement in every work-split regime, bit-reproducibility, bf16 = fp32 on widened logits,
the NaN guard for labels outside [0, K), network losses and gradients against torch's log_softmax on the same logits, CUDA
graphs, training, evaluation and launch accounting."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import rel_err

E_NULL, E_SHAPE, E_ALIGN, E_MODE, E_WORKSPACE = -1, -2, -3, -4, -5
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference
NEW = ["whvi_categorical_sizes", "whvi_categorical_nll_f32", "whvi_categorical_nll_bf16", "whvi_categorical_nll_bwd_f32",
       "whvi_categorical_nll_bwd_bf16", "whvi_categorical_predictive_f32", "whvi_categorical_predictive_bf16"]


def _nll(**kw):
    a = dict(logits=A, labels=A, lse=A, total=A, ws=A, ws_bytes=1 << 20, S=2, B=3, K=10, stream=None)
    a.update(kw)
    return tuple(a.values())


def _bwd(**kw):
    a = dict(logits=A, labels=A, lse=A, c=A, dz=A, S=2, B=3, K=10, stream=None)
    a.update(kw)
    return tuple(a.values())


def _pred(**kw):
    a = dict(logits=A, stride=30, labels=A, prob=A, ll=A, S=2, B=3, K=10, flags=0, stream=None)
    a.update(kw)
    return tuple(a.values())


# (entry point suffix, args, code, message fragment); every case fails validation, so no CUDA call is made
CASES = [
    ("nll", _nll(K=1), E_SHAPE, "outside [2, 65536]"),
    ("nll", _nll(K=65537), E_SHAPE, "outside [2, 65536]"),
    ("nll", _nll(S=-1), E_SHAPE, "S=-1"),
    ("nll", _nll(B=-3), E_SHAPE, "B=-3"),
    ("nll", _nll(logits=None), E_NULL, "null pointer"),
    ("nll", _nll(labels=None), E_NULL, "null pointer"),
    ("nll", _nll(total=None), E_NULL, "null pointer"),
    ("nll", _nll(labels=A + 4), E_ALIGN, "aligned"),
    ("nll", _nll(lse=A + 2), E_ALIGN, "aligned"),
    ("nll", _nll(total=A + 1), E_ALIGN, "aligned"),
    ("nll", _nll(ws=None), E_WORKSPACE, "workspace of 8 bytes"),
    ("nll", _nll(ws_bytes=4), E_WORKSPACE, "4 given"),
    ("nll", _nll(ws=A + 4), E_WORKSPACE, "8-byte aligned"),
    ("nll_bwd", _bwd(K=1), E_SHAPE, "outside [2, 65536]"),
    ("nll_bwd", _bwd(S=-2), E_SHAPE, "S=-2"),
    ("nll_bwd", _bwd(dz=None), E_NULL, "null pointer"),
    ("nll_bwd", _bwd(lse=None), E_NULL, "null pointer"),
    ("nll_bwd", _bwd(labels=None), E_NULL, "null pointer"),
    ("nll_bwd", _bwd(c=A + 2), E_ALIGN, "aligned"),
    ("nll_bwd", _bwd(lse=A + 1), E_ALIGN, "aligned"),
    ("predictive", _pred(K=70000), E_SHAPE, "outside [2, 65536]"),
    ("predictive", _pred(flags=2), E_MODE, "unknown flags"),
    ("predictive", _pred(stride=29), E_SHAPE, "sample_stride"),
    ("predictive", _pred(ll=None), E_NULL, "both be given"),
    ("predictive", _pred(labels=None), E_NULL, "both be given"),
    ("predictive", _pred(prob=None), E_NULL, "null pointer"),
    ("predictive", _pred(logits=None), E_NULL, "null pointer"),
    ("predictive", _pred(prob=A + 2), E_ALIGN, "aligned"),
    ("predictive", _pred(labels=A + 4), E_ALIGN, "aligned"),
]


def test_new_symbols_declared_exported_and_counted():
    from test_abi import declared_symbols
    from whvi_b200 import _lib
    from whvi_b200 import functional as WF
    L = ctypes.CDLL(str(_lib.LIB_PATH))
    declared = declared_symbols()
    for name in NEW:
        assert name in declared and hasattr(L, name) and name in _lib.SIGNATURES, name
        if name != "whvi_categorical_sizes":
            assert name in WF._LAUNCHES_PER_CALL, name
    assert WF._LAUNCHES_PER_CALL["whvi_categorical_nll_f32"] == 2   # row kernel + fixed-order total


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_validation_codes_and_messages_shim_equals_ctypes(dtype):
    from whvi_b200 import _lib
    L = _lib.lib()
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    for kind, args, code, msg in CASES:
        name = f"whvi_categorical_{kind}_{dtype}"
        fast = getattr(L, name)
        assert not hasattr(fast, "argtypes"), name          # handed out behind the shim
        rc_fast, msg_fast = fast(*args), L.whvi_last_error().decode()
        rc_raw, msg_raw = getattr(L._cdll, name)(*args), L.whvi_last_error().decode()
        assert rc_fast == rc_raw == code, (name, args, rc_fast, rc_raw, msg_fast)
        assert msg_fast == msg_raw and msg in msg_fast and name[5:] in msg_fast, (name, msg_fast)
    # bf16 logits need 2-byte alignment only, fp32 logits 4
    rc = getattr(L, f"whvi_categorical_nll_{dtype}")(*_nll(logits=A + 1))
    assert rc == E_ALIGN
    # empty problems are valid no-ops that need no pointers (no launch for the backward and the predictive)
    assert getattr(L, f"whvi_categorical_nll_bwd_{dtype}")(*_bwd(logits=None, labels=None, lse=None, dz=None, S=0)) == 0
    assert getattr(L, f"whvi_categorical_predictive_{dtype}")(*_pred(logits=None, labels=None, ll=None, prob=None, B=0)) == 0


def test_workspace_query():
    from whvi_b200 import _lib
    L = _lib.lib()
    assert hasattr(L.whvi_categorical_sizes, "argtypes")   # output pointer: stays on ctypes
    ws = ctypes.c_size_t(0)
    assert L.whvi_categorical_sizes(6, 10, ctypes.byref(ws)) == 0 and ws.value == 8
    assert L.whvi_categorical_sizes(0, 10, ctypes.byref(ws)) == 0 and ws.value == 8
    assert L.whvi_categorical_sizes(10 ** 7, 1000, ctypes.byref(ws)) == 0 and 8 < ws.value <= 8 * 148 * 16
    assert L.whvi_categorical_sizes(6, 1, ctypes.byref(ws)) == E_SHAPE
    assert L.whvi_categorical_sizes(-1, 10, ctypes.byref(ws)) == E_SHAPE
    assert L.whvi_categorical_sizes(6, 10, None) == E_NULL


# fp64 numpy restatement of the likelihood.  Not in the reference (its networks only regress): parity unpinned, tied to torch's
# cross_entropy / logsumexp / softmax and autograd by test_restatement_equals_torch_fp64.  z: (S, B, K) logits, y: (B,) labels; a
# label outside [0, K) gives NaN in its rows.
def ref_lse(z) -> np.ndarray:
    """log sum_k exp(z[..., k]), max-subtracted, fp64."""
    z = np.asarray(z, dtype=np.float64)
    m = z.max(axis=-1, keepdims=True)
    return (m + np.log(np.exp(z - m).sum(axis=-1, keepdims=True)))[..., 0]


def _label_logit(z, y):
    y = np.asarray(y, dtype=np.int64)
    K = z.shape[-1]
    ok = (y >= 0) & (y < K)
    zy = np.take_along_axis(z, np.broadcast_to(np.where(ok, y, 0)[None, :, None], z.shape[:-1] + (1,)), axis=-1)[..., 0]
    return np.where(ok[None, :], zy, np.nan)


def ref_nll(z, y):
    """(sum_{s,b} -log softmax(z[s, b])[y_b], lse (S, B), row losses (S, B)); the row loss is lse - z_y, never log of p."""
    z = np.asarray(z, dtype=np.float64)
    lse = ref_lse(z)
    rows = lse - _label_logit(z, y)
    return float(rows.sum()), lse, rows


def ref_nll_bwd(z, y, c: float = 1.0) -> np.ndarray:
    """d/dz of c * sum -log softmax(z)[y]: c (softmax(z) - onehot(y)); NaN rows for labels outside [0, K)."""
    z = np.asarray(z, dtype=np.float64)
    y = np.asarray(y, dtype=np.int64)
    K = z.shape[-1]
    ok = (y >= 0) & (y < K)
    onehot = (np.arange(K)[None, :] == y[:, None]).astype(np.float64)
    dz = c * (np.exp(z - ref_lse(z)[..., None]) - onehot[None])
    dz[:, ~ok, :] = np.nan
    return dz


def ref_predictive(z, y=None):
    """(sum_s softmax(z[s]) (B, K), sum_s log softmax(z[s])[y] (B,) or None)."""
    z = np.asarray(z, dtype=np.float64)
    lse = ref_lse(z)
    prob = np.exp(z - lse[..., None]).sum(axis=0)
    return prob, (None if y is None else (_label_logit(z, y) - lse).sum(axis=0))


def _logits(rng, S, B, K, big_rows=True):
    z = rng.standard_normal((S, B, K)) * 3.0
    if big_rows:
        z[:, 1::5] = rng.uniform(-100.0, 100.0, size=z[:, 1::5].shape)   # magnitude ~100: confident, often wrong
    return z


@pytest.mark.parametrize("K", [2, 3, 10, 33, 1000])
def test_restatement_equals_torch_fp64(K):
    rng = np.random.default_rng(K)
    S, B = 3, 41
    z = _logits(rng, S, B, K)
    y = rng.integers(0, K, size=B)
    c = 0.37
    total, lse, rows = ref_nll(z, y)
    zt = torch.from_numpy(z).requires_grad_()
    yt = torch.from_numpy(y)
    ref = F.cross_entropy(zt.reshape(S * B, K), yt.repeat(S), reduction="sum")
    (c * ref).backward()
    assert abs(total - ref.item()) <= 1e-12 * abs(ref.item())
    assert rel_err(lse, torch.logsumexp(zt.detach(), -1).numpy()) <= 1e-12
    assert rel_err(rows, -torch.log_softmax(zt.detach(), -1).gather(-1, yt.reshape(1, B, 1).expand(S, B, 1))[..., 0].numpy()) <= 1e-12
    assert rel_err(ref_nll_bwd(z, y, c), zt.grad.numpy()) <= 1e-12
    prob, ll = ref_predictive(z, y)
    p = torch.softmax(torch.from_numpy(z), -1)
    assert rel_err(prob, p.sum(0).numpy()) <= 1e-12
    assert rel_err(ll, torch.log_softmax(torch.from_numpy(z), -1).gather(-1, yt.reshape(1, B, 1).expand(S, B, 1))[..., 0].sum(0).numpy()) <= 1e-12


def test_restatement_bad_labels_are_nan_rows():
    rng = np.random.default_rng(1)
    z = _logits(rng, 2, 6, 5)
    y = np.array([0, -1, 4, 5, 2, 1])
    total, lse, rows = ref_nll(z, y)
    assert np.isnan(total) and np.isfinite(lse).all()
    assert np.isnan(rows[:, [1, 3]]).all() and np.isfinite(rows[:, [0, 2, 4, 5]]).all()
    dz = ref_nll_bwd(z, y)
    assert np.isnan(dz[:, [1, 3]]).all() and np.isfinite(dz[:, [0, 2, 4, 5]]).all()
    _, ll = ref_predictive(z, y)
    assert np.isnan(ll[[1, 3]]).all() and np.isfinite(ll[[0, 2, 4, 5]]).all()


def test_front_end_rejects_bad_inputs_without_fallback():
    from whvi_b200 import functional as WF
    z = torch.randn(2, 3, 4)
    y = torch.tensor([0, 1, 2])
    with pytest.raises(RuntimeError, match="CUDA"):
        WF.categorical_nll(z, y)
    with pytest.raises(RuntimeError, match="int64"):
        WF.categorical_nll(z, y.to(torch.int32))
    with pytest.raises(RuntimeError, match="labels must be"):
        WF.categorical_nll(z, torch.tensor([0, 1]))
    with pytest.raises(RuntimeError, match=r"\(S, B, K\)"):
        WF.categorical_nll(z[0], y)
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        WF.categorical_nll(z.double(), y)
    prob = torch.empty(3, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        WF.categorical_predictive_(z, None, prob)
    with pytest.raises(RuntimeError, match="int64"):
        WF.categorical_predictive_(z, y.to(torch.int32), prob, torch.empty(3))
    with pytest.raises(RuntimeError, match="labels must be"):
        WF.categorical_predictive_(z, torch.tensor([0]), prob, torch.empty(3))
    with pytest.raises(RuntimeError, match="CUDA"):
        WF.categorical_predictive_(z, y, prob, torch.empty(3))


def test_state_dict_has_no_likelihood_entries():
    import whvi_b200 as W
    torch.manual_seed(0)
    net = W.WHVIClassification([W.WHVILinear(8, 16), nn.ReLU(), W.WHVILinear(16, 3)])
    assert isinstance(net.likelihood, W.CategoricalLikelihood) and list(net.likelihood.parameters()) == []
    keys = list(net.state_dict().keys())
    assert keys and all(k.startswith("sequential.") for k in keys)
    assert keys == ["sequential." + k for k in net.sequential.state_dict().keys()]


def test_reduce_predictive_probs_single_process():
    from whvi_b200.distributed import reduce_predictive_probs
    prob_sum, ll = torch.rand(5, 3) * 4, -torch.rand(5) * 4
    mean, mean_ll = reduce_predictive_probs(prob_sum.clone(), ll.clone(), 4)
    assert torch.allclose(mean, prob_sum / 4) and torch.allclose(mean_ll, ll / 4)
    assert reduce_predictive_probs(prob_sum.clone(), None, 4)[1] is None


# ------------------------------------------------------------------------------------------------------------------ GPU
def dev():
    return torch.device("cuda:0")


def _raw(name, *args):
    from whvi_b200 import _lib
    rc = getattr(_lib.lib(), name)(*args)
    _lib.check(rc, name)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _run_kernels(zt, yt, c, pred_samples=None, fill=float("nan")):
    """The three entry points on device tensors with every output and the workspace prefilled (NaN by default)."""
    from whvi_b200 import functional as WF
    S, B, K = zt.shape
    sfx = "bf16" if zt.dtype == torch.bfloat16 else "f32"
    lse = torch.full((S, B), fill, device=dev())
    total = torch.full((1,), fill, device=dev())
    ws = torch.full((WF._query("whvi_categorical_sizes", S * B, K)[0] // 8,), fill, dtype=torch.float64, device=dev())
    _raw(f"whvi_categorical_nll_{sfx}", zt.data_ptr(), yt.data_ptr(), lse.data_ptr(), total.data_ptr(), ws.data_ptr(), ws.numel() * 8,
         S, B, K, _stream())
    dz = torch.full_like(zt, fill)
    _raw(f"whvi_categorical_nll_bwd_{sfx}", zt.data_ptr(), yt.data_ptr(), lse.data_ptr(), c.data_ptr(), dz.data_ptr(), S, B, K, _stream())
    prob = torch.full((B, K), fill, device=dev())
    ll = torch.full((B,), fill, device=dev())
    _raw(f"whvi_categorical_predictive_{sfx}", zt.data_ptr(), B * K, yt.data_ptr(), prob.data_ptr(), ll.data_ptr(), S, B, K, 0, _stream())
    return total, lse, dz, prob, ll


# rows per CTA pass: 256 / TPR groups; 148 * 16 CTAs before the grid strides.  The row counts below give a partial last CTA,
# more than one wave, and (K <= 4096) more rows than one pass of the capped grid
ROWS = {2: 303333, 3: 151653, 10: 38002, 17: 19002, 100: 19002, 1000: 19002, 4096: 2402, 65536: 1202}


@pytest.mark.gpu
@pytest.mark.parametrize("K", sorted(ROWS))
def test_kernels_against_fp64_restatement(K):
    rng = np.random.default_rng(K)
    S = 2
    B = ROWS[K] // S
    z = _logits(rng, S, B, K).astype(np.float32)
    y = rng.integers(0, K, size=B)
    zt, yt = torch.from_numpy(z).to(dev()), torch.from_numpy(y).to(dev())
    c = torch.tensor([0.37], device=dev())
    total, lse, dz, prob, ll = _run_kernels(zt, yt, c)
    torch.cuda.synchronize()
    ref_total, ref_lse, _ = ref_nll(z, y)
    assert abs(total.item() - ref_total) <= 1e-5 * abs(ref_total)
    assert rel_err(lse.cpu().numpy(), ref_lse) <= 1e-5
    assert rel_err(dz.cpu().numpy(), ref_nll_bwd(z, y, 0.37)) <= 1e-5
    ref_prob, ref_ll = ref_predictive(z, y)
    assert rel_err(prob.cpu().numpy(), ref_prob) <= 1e-5
    assert rel_err(ll.cpu().numpy(), ref_ll) <= 1e-5
    # bit-reproducible, and independent of what the buffers held
    again = _run_kernels(zt, yt, c, fill=0.0)
    for a, b in zip((total, lse, dz, prob, ll), again):
        assert torch.equal(a, b)
    # ACCUMULATE over two sample chunks (strided views of the same tensor) equals one call over all samples
    prob2, ll2 = torch.full_like(prob, float("nan")), torch.full_like(ll, float("nan"))
    for s0, s1 in ((0, 1), (1, S)):
        _raw("whvi_categorical_predictive_f32", zt[s0:s1].data_ptr(), B * K, yt.data_ptr(), prob2.data_ptr(), ll2.data_ptr(), s1 - s0,
             B, K, 1 if s0 else 0, _stream())
    assert torch.equal(prob2, prob) and torch.equal(ll2, ll)
    # bf16: the fp32 kernels on the widened logits, bit for bit; dz rounded once
    zb = zt.to(torch.bfloat16)
    wide = _run_kernels(zb.float(), yt, c)
    got = _run_kernels(zb, yt, c)
    for i, (a, b) in enumerate(zip(got, wide)):
        assert torch.equal(a, b.to(torch.bfloat16) if i == 2 else b), i


@pytest.mark.gpu
def test_bf16_beyond_2_31_elements():
    """S * B * K > 2^31 (int64 indexing everywhere): the total against torch fp64 in row chunks, the last rows (past element
    2^31) against the fp64 restatement."""
    S, B, K = 2, 16385, 65536
    assert S * B * K > 2 ** 31
    g = torch.Generator(device=dev()).manual_seed(5)
    zb = (torch.randn((S, B, K), device=dev(), generator=g) * 3).to(torch.bfloat16)
    yt = torch.randint(0, K, (B,), device=dev(), generator=g)
    c = torch.tensor([1.5], device=dev())
    total, lse, dz, prob, ll = _run_kernels(zb, yt, c)
    ref = 0.0
    flat, ys = zb.reshape(S * B, K), yt.repeat(S)
    for r0 in range(0, S * B, 2048):
        zc = flat[r0:r0 + 2048].double()
        ref += float((torch.logsumexp(zc, -1) - zc.gather(1, ys[r0:r0 + 2048, None])[:, 0]).sum())
    assert abs(total.item() - ref) <= 1e-5 * abs(ref)
    tail = zb[:, -3:].float().cpu().numpy()
    ytail = yt[-3:].cpu().numpy()
    assert rel_err(lse[:, -3:].cpu().numpy(), ref_lse(tail)) <= 1e-5
    assert rel_err(dz[:, -3:].float().cpu().numpy(), ref_nll_bwd(tail, ytail, 1.5)) <= 1e-2   # bf16 dz: 8 bits
    ref_prob, ref_ll = ref_predictive(tail, ytail)
    assert rel_err(prob[-3:].cpu().numpy(), ref_prob) <= 1e-5 and rel_err(ll[-3:].cpu().numpy(), ref_ll) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 1000, 4096])
def test_labels_outside_range_give_nan_rows_only(K):
    rng = np.random.default_rng(3)
    S, B = 3, 37
    zt = torch.from_numpy(_logits(rng, S, B, K).astype(np.float32)).to(dev())
    y = rng.integers(0, K, size=B)
    good = torch.from_numpy(y).to(dev())
    bad_rows = [5, 20]   # interior: an unguarded read of label -1 or K lands inside the tensor, as a wrong number
    y[bad_rows[0]], y[bad_rows[1]] = -1, K
    bad = torch.from_numpy(y).to(dev())
    c = torch.tensor([1.0], device=dev())
    t0, lse0, dz0, prob0, ll0 = _run_kernels(zt, good, c)
    t1, lse1, dz1, prob1, ll1 = _run_kernels(zt, bad, c)
    keep = [b for b in range(B) if b not in bad_rows]
    assert torch.isfinite(t0).all() and torch.isnan(t1).all()
    assert torch.equal(lse1, lse0) and torch.equal(prob1, prob0)
    assert torch.isnan(dz1[:, bad_rows]).all() and torch.equal(dz1[:, keep], dz0[:, keep])
    assert torch.isnan(ll1[bad_rows]).all() and torch.equal(ll1[keep], ll0[keep])


# ------------------------------------------------------------------------------------------------------------------ networks
def _net(kind, seed=0):
    import whvi_b200 as W
    torch.manual_seed(seed)
    if kind == "stacked":
        mods, d_in, K = [W.WHVILinear(64, 128, bias=True), nn.ReLU(), W.WHVILinear(128, 10, bias=True)], 64, 10
    elif kind == "square":
        mods, d_in, K = [W.WHVILinear(256, 1024), nn.ReLU(), W.WHVILinear(1024, 1024, bias=True)], 256, 1024
    elif kind == "linear":
        mods, d_in, K = [W.WHVILinear(64, 64, bias=True), nn.ReLU(), nn.Linear(64, 5)], 64, 5
    elif kind == "dense":
        mods, d_in, K = [W.WHVILinear(64, 128, covariance="dense"), nn.ReLU(), W.WHVILinear(128, 7, covariance="dense")], 64, 7
    else:
        raise ValueError(kind)
    net = W.WHVIClassification(mods, train_samples=4, eval_samples=8).to(dev())
    with torch.no_grad():   # a posterior with visible noise, so eps matters
        for name, p in net.named_parameters():
            if name.endswith("g_mu"):
                p.normal_()
    return net, d_in, K


def _inject(net, S, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    for layer in net._whvi_layers():
        for blk in layer.square_blocks():
            blk.inject_eps(torch.randn((S, blk.D), device=dev(), generator=g))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,bf16", [("stacked", False), ("square", False), ("linear", False), ("dense", False), ("stacked", True),
                                       ("square", True)])
def test_network_loss_and_gradients_match_torch_log_softmax(kind, bf16):
    net, d_in, K = _net(kind)
    S, B, n = net.train_samples, 48, 1000
    g = torch.Generator(device=dev()).manual_seed(1)
    x = torch.randn((B, d_in), device=dev(), generator=g)
    if bf16:
        x = x.to(torch.bfloat16)
    y = torch.randint(0, K, (B,), device=dev(), generator=g)
    ref = copy.deepcopy(net)
    _inject(net, S, 7)
    loss = net.loss(x, y, n=n)
    loss.backward()
    _inject(ref, S, 7)
    logits = ref._run(x, S)
    assert logits.shape == (S, B, K) and logits.dtype == (torch.bfloat16 if bf16 and kind != "linear" else torch.float32)
    lp = torch.log_softmax(logits.double(), -1).gather(-1, y.reshape(1, B, 1).expand(S, B, 1))
    ref_loss = -(n / (B * S)) * lp.sum() + ref.kl
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    for (name, p), q in zip(net.named_parameters(), ref.parameters()):
        assert p.grad is not None and q.grad is not None, name
        assert rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) <= 1e-5, name


def _blobs(n, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    centres = torch.tensor([[2.0, 0.0], [-1.0, 1.7], [-1.0, -1.7]], device=dev())
    y = torch.randint(0, 3, (n,), device=dev(), generator=g)
    x = centres[y] + 0.5 * torch.randn((n, 2), device=dev(), generator=g)
    return torch.cat([x, torch.zeros((n, 14), device=dev())], 1), y


def _blob_net(seed=0):
    import whvi_b200 as W
    torch.manual_seed(seed)
    return W.WHVIClassification([W.WHVILinear(16, 64, lambda_=1.0, bias=True), nn.ReLU(), W.WHVILinear(64, 3, lambda_=1.0, bias=True)],
                                train_samples=2, eval_samples=16).to(dev())


@pytest.mark.gpu
def test_cuda_graph_step_equals_eager_step():
    """Posterior noise off (softplus(-30) ~ 1e-13 next to O(1) means), so both runs see the same weights."""
    from whvi_b200 import FlatAdam, FlatParams
    from whvi_b200.graphs import GraphedTrainStep
    eager = _blob_net()
    with torch.no_grad():
        for name, p in eager.named_parameters():
            if name.endswith("g_mu"):
                p.normal_()
            if name.endswith("g_rho"):
                p.fill_(-30.0)
    graphed = copy.deepcopy(eager)
    opt_e = FlatAdam(FlatParams(eager.parameters()), lr=1e-2)
    opt_g = FlatAdam(FlatParams(graphed.parameters()), lr=1e-2)
    batches = [_blobs(32, s) for s in range(3)]
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
def test_train_model_cuda_graph_learns_three_blobs():
    from whvi_b200 import FlatAdam, FlatParams
    net = _blob_net()
    x, y = _blobs(512, 0)
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(x, y), batch_size=64, shuffle=False)
    opt = FlatAdam(FlatParams(net.parameters()), lr=torch.tensor(1e-2, device=dev()))
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda _: 1.0)
    net.train_model(loader, opt, sched, epochs1=30, epochs2=30, cuda_graph=True)
    xt, yt = _blobs(1024, 1)
    err, mnll = net.eval_model(xt, yt)
    assert err <= 0.10 and mnll == mnll, (err, mnll)
    assert (net.predict_proba(xt).argmax(1) == yt).float().mean().item() >= 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["stacked", "linear"])
def test_eval_model_equals_fp64_from_forward(kind):
    net, d_in, K = _net(kind)
    net.eval()
    S, B = net.eval_samples, 300
    g = torch.Generator(device=dev()).manual_seed(2)
    x = torch.randn((B, d_in), device=dev(), generator=g)
    y = torch.randint(0, K, (B,), device=dev(), generator=g)
    _inject(net, S, 11)
    y_pred = net(x)                                       # (B, K, S)
    lp = torch.log_softmax(y_pred.double(), 1)
    ref_err = float((lp.exp().mean(2).argmax(1) != y).double().mean())
    ref_mnll = float(-lp.gather(1, y.reshape(B, 1, 1).expand(B, 1, S)).sum() / S)
    assert S <= 16   # eval_model runs 16 samples at a time: one chunk, so one injection gives it forward()'s noise
    _inject(net, S, 11)
    err, mnll = net.eval_model(x, y)
    assert err == ref_err
    assert abs(mnll - ref_mnll) <= 1e-5 * abs(ref_mnll)
    # a user loss gets the (B, K, S) logits of forward()
    _inject(net, S, 11)
    seen = {}
    err2, mnll2 = net.eval_model(x, y, loss=lambda yp, yt: seen.setdefault("shape", tuple(yp.shape)) and 0.0)
    assert seen["shape"] == (B, K, S) and abs(mnll2 - ref_mnll) <= 1e-5 * abs(ref_mnll)


@pytest.mark.gpu
def test_chunked_predict_proba_equals_one_kernel_call():
    from whvi_b200 import functional as WF
    net, d_in, K = _net("stacked")
    net.eval()
    S, B, chunk = 7, 50, 3
    x = torch.randn((B, d_in), device=dev())
    chunks = [(s0, min(S, s0 + chunk)) for s0 in range(0, S, chunk)]
    for i, (s0, s1) in enumerate(chunks):
        _inject(net, s1 - s0, 100 + i)
    proba = net.predict_proba(x, n_samples=S, chunk_samples=chunk)
    logits = []
    for i, (s0, s1) in enumerate(chunks):
        _inject(net, s1 - s0, 100 + i)
        logits.append(net._run(x, s1 - s0))
    prob_sum = torch.empty((B, K), device=dev())
    WF.categorical_predictive_(torch.cat(logits), None, prob_sum)
    assert torch.equal(proba, prob_sum / S)
    assert torch.allclose(proba.sum(1), torch.ones(B, device=dev()), atol=1e-5)


@pytest.mark.gpu
def test_classification_step_adds_exactly_the_likelihood_launches():
    from whvi_b200 import functional as WF
    net, d_in, K = _net("stacked")
    x = torch.randn((16, d_in), device=dev())
    y = torch.randint(0, K, (16,), device=dev())

    def count(fn):
        WF.LAUNCH_COUNTS.clear()
        fn()
        out = dict(WF.LAUNCH_COUNTS)
        WF.LAUNCH_COUNTS.clear()
        return out

    layers = count(lambda: (net._run(x, net.train_samples).float().sum() + net.kl).backward())
    step = count(lambda: net.loss(x, y, n=100).backward())
    extra = {k: step.get(k, 0) - layers.get(k, 0) for k in set(step) | set(layers)}
    assert {k: v for k, v in extra.items() if v} == {"whvi_categorical_nll_f32": 2, "whvi_categorical_nll_bwd_f32": 1}
