"""Class weights, label smoothing and ignore_index for classifiers: the options instances of the sm_100a cross-entropy kernels
(``csrc/categorical.cu``, ``whvi_categorical_nll_ex_*`` / ``whvi_categorical_nll_bwd_ex_*``) up to ``CategoricalLikelihood`` and
``WHVIClassification``.

CPU: an fp64 numpy restatement of the loss and its gradient tied to torch's fp64 ``F.cross_entropy(..., reduction="sum")`` and its
autograd; validation codes and messages of the four entry points; bindings and launch counts; the likelihood's and network's
constructor checks and an unchanged state_dict.
GPU: the kernels against the restatement in every work-split regime (partial last row groups, more rows than one pass of the
grid), outputs and workspace filled with NaN first, logits offset by 1e3, NaN rows for labels outside [0, K) next to zero rows
for ignored ones, bit-reproducibility, bf16 = fp32 on widened logits; the networks against torch fp64 cross_entropy on their own
logits, a CUDA-graph step, evaluation over the labelled rows and launch accounting."""
import copy
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from conftest import rel_err

E_NULL, E_SHAPE, E_ALIGN, E_MODE, E_WORKSPACE = -1, -2, -3, -4, -5
IGNORE = 2   # WHVI_CATEGORICAL_IGNORE
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference
NEW = ["whvi_categorical_nll_ex_f32", "whvi_categorical_nll_ex_bf16", "whvi_categorical_nll_bwd_ex_f32",
       "whvi_categorical_nll_bwd_ex_bf16"]


# fp64 numpy restatement.  z: (S, B, K) logits, y: (B,) labels, w: (K,) weights or None (ones), eps: label smoothing,
# ignore: ignore_index or None.  An ignored row gives 0 and a zero dz row; any other label outside [0, K) gives NaN.
def ref_lse(z):
    m = z.max(axis=-1, keepdims=True)
    return (m + np.log(np.exp(z - m).sum(axis=-1, keepdims=True)))[..., 0]


def _masks(y, K, ignore):
    y = np.asarray(y, dtype=np.int64)
    ign = np.zeros(y.shape, bool) if ignore is None else y == ignore
    ok = (y >= 0) & (y < K)
    return y, ign, ok


def ref_loss(z, y, w=None, eps=0.0, ignore=None):
    """(total, row losses (S, B)): (1 - eps) w_y (lse - z_y) + (eps / K) sum_k w_k (lse - z_k)."""
    z = np.asarray(z, dtype=np.float64)
    K = z.shape[-1]
    w = np.ones(K) if w is None else np.asarray(w, dtype=np.float64)
    y, ign, ok = _masks(y, K, ignore)
    lse = ref_lse(z)
    yc = np.where(ok, y, 0)
    zy = np.take_along_axis(z, np.broadcast_to(yc[None, :, None], z.shape[:-1] + (1,)), axis=-1)[..., 0]
    rows = (1 - eps) * w[yc][None] * (lse - zy) + (eps / K) * (w * (lse[..., None] - z)).sum(-1)
    rows = np.where(ok[None], rows, np.nan)
    rows = np.where(ign[None], 0.0, rows)
    return float(rows.sum()), rows


def ref_grad(z, y, w=None, eps=0.0, ignore=None, c=1.0):
    """dz = c [(1 - eps) w_y (p - onehot(y)) + (eps / K) (W p - w)]."""
    z = np.asarray(z, dtype=np.float64)
    K = z.shape[-1]
    w = np.ones(K) if w is None else np.asarray(w, dtype=np.float64)
    y, ign, ok = _masks(y, K, ignore)
    yc = np.where(ok, y, 0)
    p = np.exp(z - ref_lse(z)[..., None])
    onehot = (np.arange(K)[None, :] == yc[:, None]).astype(np.float64)
    dz = c * ((1 - eps) * w[yc][None, :, None] * (p - onehot[None]) + (eps / K) * (w.sum() * p - w))
    dz[:, ~ok] = np.nan
    dz[:, ign] = 0.0
    return dz


def _logits(rng, S, B, K):
    z = rng.standard_normal((S, B, K)) * 3.0
    z[:, 1::5] = rng.uniform(-100.0, 100.0, size=z[:, 1::5].shape)   # confident, often wrong rows
    return z


def _weights(rng, kind, K):
    if kind == "none":
        return None
    w = rng.uniform(0.1, 3.0, size=K)
    if kind == "zeros":
        w[::3] = 0.0
    return w


def _labels(rng, kind, B, K):
    """(labels, ignore_index) for an ignore setting: off, -100, an in-range class, or every row ignored."""
    y = rng.integers(0, K, size=B)
    if kind == "off":
        return y, None
    if kind == "-100":
        y[::4] = -100
        return y, -100
    if kind == "class":
        y[::3] = 1
        return y, 1
    return np.full(B, K - 1), K - 1   # "all"


EPS = [0.0, 0.1, 1.0]
WEIGHTS = ["none", "random", "zeros"]
IGNORES = ["off", "-100", "class", "all"]


@pytest.mark.parametrize("K", [2, 5, 33])
@pytest.mark.parametrize("eps", EPS)
@pytest.mark.parametrize("wk", WEIGHTS)
@pytest.mark.parametrize("ik", IGNORES)
def test_restatement_equals_torch_fp64(K, eps, wk, ik):
    rng = np.random.default_rng(K * 100 + EPS.index(eps) * 10 + WEIGHTS.index(wk) + 1000 * IGNORES.index(ik))
    S, B = 3, 23
    z = _logits(rng, S, B, K)
    w = _weights(rng, wk, K)
    y, ignore = _labels(rng, ik, B, K)
    c = 0.37
    total, rows = ref_loss(z, y, w, eps, ignore)
    zt = torch.from_numpy(z).requires_grad_()
    kw = dict(weight=None if w is None else torch.from_numpy(w), label_smoothing=eps, reduction="sum")
    if ignore is not None:
        kw["ignore_index"] = ignore
    ref = F.cross_entropy(zt.reshape(S * B, K), torch.from_numpy(y).repeat(S), **kw)
    (c * ref).backward()
    assert abs(total - ref.item()) <= 1e-12 * max(abs(ref.item()), 1.0)
    assert rel_err(ref_grad(z, y, w, eps, ignore, c), zt.grad.numpy()) <= 1e-12
    if ignore is not None:
        assert np.all(rows[:, y == ignore] == 0.0)
    if ik == "all":
        assert total == 0.0 and not ref_grad(z, y, w, eps, ignore, c).any()


def test_restatement_bad_labels_and_ignored_rows():
    rng = np.random.default_rng(1)
    K = 5
    z = _logits(rng, 2, 6, K)
    y = np.array([0, -1, -100, K, 2, 1])
    w = rng.uniform(0.5, 2.0, size=K)
    total, rows = ref_loss(z, y, w, 0.1, -100)
    assert np.isnan(total) and np.isnan(rows[:, [1, 3]]).all() and (rows[:, 2] == 0).all() and np.isfinite(rows[:, [0, 4, 5]]).all()
    dz = ref_grad(z, y, w, 0.1, -100)
    assert np.isnan(dz[:, [1, 3]]).all() and (dz[:, 2] == 0).all() and np.isfinite(dz[:, [0, 4, 5]]).all()
    # without ignore_index, -100 is just a label outside [0, K)
    assert np.isnan(ref_loss(z, y, w, 0.1, None)[1][:, 2]).all()


def test_new_symbols_declared_exported_and_counted():
    from test_abi import declared_symbols
    from whvi_b200 import _lib
    from whvi_b200 import functional as WF
    L = ctypes.CDLL(str(_lib.LIB_PATH))
    declared = declared_symbols()
    for name in NEW:
        assert name in declared and hasattr(L, name) and name in _lib.SIGNATURES, name
        assert WF._LAUNCHES_PER_CALL[name] == (1 if "_bwd_" in name else 2), name
        assert hasattr(getattr(_lib.lib(), name), "argtypes"), name   # a float parameter: stays on ctypes
    assert WF.CATEGORICAL_IGNORE == IGNORE


def _nll(**kw):
    a = dict(logits=A, labels=A, lse=A, total=A, ws=A, ws_bytes=1 << 20, S=2, B=3, K=10, w=A, eps=0.1, ignore_index=-100,
             flags=IGNORE, stream=None)
    a.update(kw)
    return tuple(a.values())


def _bwd(**kw):
    a = dict(logits=A, labels=A, lse=A, c=A, dz=A, S=2, B=3, K=10, w=A, eps=0.1, ignore_index=-100, flags=IGNORE, stream=None)
    a.update(kw)
    return tuple(a.values())


# (entry point, args, code, message fragment); every case fails validation, so no CUDA call is made
CASES = [(kind, mk(**kw), code, msg) for kind, mk in (("nll_ex", _nll), ("nll_bwd_ex", _bwd)) for kw, code, msg in (
    (dict(eps=-0.1), E_SHAPE, "label_smoothing = -0.1 outside [0, 1]"),
    (dict(eps=1.5), E_SHAPE, "outside [0, 1]"),
    (dict(eps=float("nan")), E_SHAPE, "outside [0, 1]"),
    (dict(eps=float("inf")), E_SHAPE, "outside [0, 1]"),
    (dict(flags=1), E_MODE, "unknown flags 1"),
    (dict(flags=IGNORE | 4), E_MODE, "unknown flags 6"),
    (dict(w=A + 2), E_ALIGN, "weight must be 4-byte aligned"),
    (dict(K=1), E_SHAPE, "outside [2, 65536]"),
    (dict(K=65537, eps=2.0), E_SHAPE, "K = 65537"),        # the plain checks come first
    (dict(S=-1), E_SHAPE, "S=-1"),
    (dict(logits=None), E_NULL, "null pointer"),
    (dict(labels=None), E_NULL, "null pointer"),
    (dict(labels=A + 4), E_ALIGN, "aligned"),
    (dict(lse=A + 2), E_ALIGN, "aligned"),
)] + [
    ("nll_ex", _nll(total=None), E_NULL, "null pointer"),
    ("nll_ex", _nll(ws=None), E_WORKSPACE, "workspace of 8 bytes"),
    ("nll_ex", _nll(ws_bytes=4), E_WORKSPACE, "4 given"),
    ("nll_bwd_ex", _bwd(dz=None), E_NULL, "null pointer"),
    ("nll_bwd_ex", _bwd(c=A + 2), E_ALIGN, "aligned"),
]


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_validation_codes_and_messages(dtype):
    from whvi_b200 import _lib
    L = _lib.lib()
    for kind, args, code, msg in CASES:
        name = f"whvi_categorical_{kind}_{dtype}"
        rc = getattr(L, name)(*args)
        err = L.whvi_last_error().decode()
        assert rc == code, (name, args, rc, err)
        assert msg in err and name[5:] in err, (name, err)
    # NULL weight (ones), no flags and the ends of [0, 1] pass the option checks: the next failure is the plain null check
    for eps in (0.0, 1.0):
        assert getattr(L, f"whvi_categorical_nll_ex_{dtype}")(*_nll(w=None, eps=eps, flags=0, logits=None)) == E_NULL
    # bf16 logits need 2-byte alignment only, fp32 logits 4
    assert getattr(L, f"whvi_categorical_nll_ex_{dtype}")(*_nll(logits=A + 1)) == E_ALIGN
    # an empty problem is a valid no-op for the backward (no launch), once the options are valid
    assert getattr(L, f"whvi_categorical_nll_bwd_ex_{dtype}")(*_bwd(logits=None, labels=None, lse=None, dz=None, S=0)) == 0
    assert getattr(L, f"whvi_categorical_nll_bwd_ex_{dtype}")(*_bwd(logits=None, S=0, eps=3.0)) == E_SHAPE


def test_likelihood_and_network_constructor_checks_and_state_dict():
    import whvi_b200 as W
    from whvi_b200.likelihoods import CategoricalLikelihood
    for bad in (torch.ones(2, 3), torch.ones(1), torch.tensor([1.0, -0.5, 1.0]), torch.tensor([1.0, float("nan")]),
                torch.tensor([1.0, float("inf")])):
        with pytest.raises(ValueError, match="weight"):
            CategoricalLikelihood(weight=bad)
    for eps in (-0.01, 1.01, float("nan")):
        with pytest.raises(ValueError, match="label_smoothing"):
            CategoricalLikelihood(label_smoothing=eps)
    for ii in (1.5, True):
        with pytest.raises(ValueError, match="ignore_index"):
            CategoricalLikelihood(ignore_index=ii)
    lik = CategoricalLikelihood(weight=[1, 2, 3], label_smoothing=1, ignore_index=-100)
    assert lik.weight.dtype == torch.float32 and lik.weight.tolist() == [1.0, 2.0, 3.0]
    assert lik.label_smoothing == 1.0 and lik.ignore_index == -100
    assert lik.labelled(torch.tensor([0, -100, 2])).tolist() == [True, False, True]
    plain = CategoricalLikelihood()
    assert plain.weight is None and plain.label_smoothing == 0.0 and plain.ignore_index is None
    assert plain.labelled(torch.tensor([0, -100])) is None

    def make(**kw):
        torch.manual_seed(0)
        return W.WHVIClassification([W.WHVILinear(8, 16), nn.ReLU(), W.WHVILinear(16, 3)], **kw)

    net = make(weight=torch.tensor([1.0, 0.0, 2.0]), label_smoothing=0.1, ignore_index=-1)
    assert net.likelihood.weight.tolist() == [1.0, 0.0, 2.0] and net.likelihood.label_smoothing == 0.1
    assert net.likelihood.ignore_index == -1
    assert "likelihood.weight" in dict(net.named_buffers())
    sd, sd0 = net.state_dict(), make().state_dict()
    assert list(sd) == list(sd0) and all(torch.equal(sd[k], sd0[k]) for k in sd)   # checkpoints stay interchangeable
    make().load_state_dict(sd)
    net.load_state_dict(sd0)
    assert net.likelihood.weight.tolist() == [1.0, 0.0, 2.0]
    with pytest.raises(TypeError):
        W.WHVIClassification([W.WHVILinear(8, 3)], None)   # the options are keyword-only
    with pytest.raises(ValueError, match="label_smoothing"):
        make(label_smoothing=2.0)


def test_front_end_checks_options_before_the_device():
    from whvi_b200 import functional as WF
    assert WF._categorical_opts(torch.empty(2, 3, 4), None, 0.0, None) is None    # defaults: the plain calls
    z = torch.empty(2, 3, 4)
    for bad in (torch.ones(3), torch.ones(4, dtype=torch.float64), torch.ones(2, 4)[:, 0]):
        with pytest.raises(RuntimeError, match=r"weight must be a contiguous float32 \(4,\) tensor"):
            WF._categorical_opts(z, bad, 0.0, None)
    with pytest.raises(RuntimeError, match="label_smoothing"):
        WF._categorical_opts(z, None, 1.5, None)
    w = torch.ones(4)
    assert WF._categorical_opts(z, w, 0.25, None) == (w.data_ptr(), 0.25, 0, 0)
    assert WF._categorical_opts(z, None, 0.0, -100) == (None, 0.0, -100, IGNORE)


# ------------------------------------------------------------------------------------------------------------------ GPU
def dev():
    return torch.device("cuda:0")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _run(zt, yt, c, wt=None, eps=0.0, ignore=None, fill=float("nan")):
    """(total, lse, dz) from the two _ex entry points, every output and the workspace prefilled (NaN by default)."""
    from whvi_b200 import _lib
    from whvi_b200 import functional as WF
    L = _lib.lib()
    S, B, K = zt.shape
    sfx = "bf16" if zt.dtype == torch.bfloat16 else "f32"
    opts = (None if wt is None else wt.data_ptr(), eps, 0 if ignore is None else ignore, 0 if ignore is None else IGNORE)
    lse = torch.full((S, B), fill, device=dev())
    total = torch.full((1,), fill, device=dev())
    ws = torch.full((WF._query("whvi_categorical_sizes", S * B, K)[0] // 8,), fill, dtype=torch.float64, device=dev())
    name = f"whvi_categorical_nll_ex_{sfx}"
    _lib.check(getattr(L, name)(zt.data_ptr(), yt.data_ptr(), lse.data_ptr(), total.data_ptr(), ws.data_ptr(), ws.numel() * 8, S, B, K,
                                *opts, _stream()), name)
    dz = torch.full_like(zt, fill)
    name = f"whvi_categorical_nll_bwd_ex_{sfx}"
    _lib.check(getattr(L, name)(zt.data_ptr(), yt.data_ptr(), lse.data_ptr(), c.data_ptr(), dz.data_ptr(), S, B, K, *opts, _stream()),
               name)
    return total, lse, dz


def _t(a, dtype=None):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev()) if dtype is None else torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(dev())


# rows per CTA pass: 256 / TPR; 148 * 16 CTAs before the grid strides.  Each count leaves a partial last row group and, but for
# K = 65536, is more rows than one pass of the capped grid holds
ROWS = {2: 303333, 3: 151653, 17: 19002, 32: 19002, 33: 19002, 1000: 19002, 2048: 19002, 2049: 2402, 65536: 301}
OPTS = [("random", 0.1, "-100"), ("zeros", 1.0, "class"), ("none", 0.1, "off"), ("random", 0.0, "class")]


@pytest.mark.gpu
@pytest.mark.parametrize("K", sorted(ROWS))
def test_kernels_against_fp64_restatement(K):
    rng = np.random.default_rng(K)
    S = 2
    B = ROWS[K] // S
    z = _logits(rng, S, B, K).astype(np.float32)
    zt = _t(z)
    c = torch.tensor([0.37], device=dev())
    for i, (wk, eps, ik) in enumerate(OPTS[:2] if K >= 2048 else OPTS):
        w = _weights(rng, wk, K)
        y, ignore = _labels(rng, ik, B, K)
        wt, yt = (None if w is None else _t(w, np.float32)), _t(y)
        total, lse, dz = _run(zt, yt, c, wt, eps, ignore)
        torch.cuda.synchronize()
        w32 = None if w is None else w.astype(np.float32)
        ref_total, _ = ref_loss(z, y, w32, eps, ignore)
        assert abs(total.item() - ref_total) <= 1e-5 * abs(ref_total), (i, total.item(), ref_total)
        assert rel_err(lse.cpu().numpy(), ref_lse(z.astype(np.float64))) <= 1e-5
        assert rel_err(dz.cpu().numpy(), ref_grad(z, y, w32, eps, ignore, 0.37)) <= 1e-5, i
        # bit-reproducible, and independent of what the buffers held
        for a, b in zip((total, lse, dz), _run(zt, yt, c, wt, eps, ignore, fill=0.0)):
            assert torch.equal(a, b), i
        # bf16: the fp32 kernels on the widened logits, bit for bit; dz rounded once
        if i == 0:
            zb = zt.to(torch.bfloat16)
            wide = _run(zb.float(), yt, c, wt, eps, ignore)
            got = _run(zb, yt, c, wt, eps, ignore)
            assert torch.equal(got[0], wide[0]) and torch.equal(got[1], wide[1])
            assert torch.equal(got[2], wide[2].to(torch.bfloat16))


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 1000, 4096])
def test_option_grid_small_batches(K):
    """Every (weights, smoothing, ignore) setting on a small batch, with NULL weights for "none"."""
    rng = np.random.default_rng(7 + K)
    S, B = 3, 37
    z = _logits(rng, S, B, K).astype(np.float32)
    zt = _t(z)
    c = torch.tensor([1.25], device=dev())
    for wk in WEIGHTS:
        for eps in EPS:
            for ik in IGNORES:
                w = _weights(rng, wk, K)
                w32 = None if w is None else w.astype(np.float32)
                y, ignore = _labels(rng, ik, B, K)
                total, lse, dz = _run(zt, _t(y), c, None if w is None else _t(w32), eps, ignore)
                ref_total, _ = ref_loss(z, y, w32, eps, ignore)
                case = (wk, eps, ik)
                if ik == "all":
                    assert total.item() == 0.0 and not dz.any(), case
                else:
                    assert abs(total.item() - ref_total) <= 1e-5 * abs(ref_total), case
                    assert rel_err(dz.cpu().numpy(), ref_grad(z, y, w32, eps, ignore, 1.25)) <= 1e-5, case


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 1000, 65536])
def test_offset_logits_keep_the_smoothing_term(K):
    """Logits around 1e3: every smoothing term w_k (lse - z_k) is a difference of two numbers near 1e3 taken before the sum, so
    the total keeps fp32 accuracy (a sum_k w_k z_k subtracted from W lse would lose 2-3 digits here).  lse itself is rounded to
    ulp(1e3) = 6e-5, which bounds what dz (through p = exp(z - lse)) can reach: 1e-4."""
    rng = np.random.default_rng(K)
    S, B = 2, 301 if K == 65536 else 3001
    z = (rng.standard_normal((S, B, K)) * 3.0 + 1000.0).astype(np.float32)
    w = rng.uniform(0.1, 3.0, size=K).astype(np.float32)
    y = rng.integers(0, K, size=B)
    c = torch.tensor([1.0], device=dev())
    total, lse, dz = _run(_t(z), _t(y), c, _t(w), 0.1, None)
    ref_total, _ = ref_loss(z, y, w, 0.1, None)
    assert abs(total.item() - ref_total) <= 1e-5 * abs(ref_total), (total.item(), ref_total)
    assert rel_err(lse.cpu().numpy(), ref_lse(z.astype(np.float64))) <= 1e-6
    assert rel_err(dz.cpu().numpy(), ref_grad(z, y, w, 0.1, None)) <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 1000, 4096])
def test_bad_labels_give_nan_rows_next_to_zero_ignored_rows(K):
    rng = np.random.default_rng(3)
    S, B = 3, 37
    zt = _t(_logits(rng, S, B, K).astype(np.float32))
    wt = _t(rng.uniform(0.5, 2.0, size=K), np.float32)
    c = torch.tensor([1.0], device=dev())
    y = rng.integers(0, K, size=B)
    y[[4, 11]] = -100                      # ignored
    clean = y.copy()
    y[[5, 20]] = -1, K                     # outside [0, K), not ignored: NaN
    clean[[5, 20]] = -100
    t0, lse0, dz0 = _run(zt, _t(clean), c, wt, 0.1, -100)
    t1, lse1, dz1 = _run(zt, _t(y), c, wt, 0.1, -100)
    keep = [b for b in range(B) if b not in (5, 20)]
    assert torch.isfinite(t0).all() and torch.isnan(t1).all() and torch.equal(lse1, lse0)
    assert torch.isnan(dz1[:, [5, 20]]).all() and torch.equal(dz1[:, keep], dz0[:, keep])
    assert torch.all(dz1[:, [4, 11]] == 0.0) and torch.all(dz0[:, [4, 11, 5, 20]] == 0.0)
    # the ignore test comes before the range test, and only with the flag: without it -100 is a bad label
    t2, _, dz2 = _run(zt, _t(clean), c, wt, 0.1, None)
    assert torch.isnan(t2).all() and torch.isnan(dz2[:, [4, 11]]).all()


@pytest.mark.gpu
def test_functional_routes_and_front_end_checks():
    from whvi_b200 import functional as WF
    S, B, K = 2, 9, 6
    z = torch.randn((S, B, K), device=dev(), requires_grad=True)
    y = torch.randint(0, K, (B,), device=dev())
    with pytest.raises(RuntimeError, match="weight must be"):
        WF.categorical_nll(z, y, torch.ones(K))                                    # on the CPU
    with pytest.raises(RuntimeError, match="weight must be"):
        WF.categorical_nll(z, y, torch.ones(K + 1, device=dev()))

    def launches(**kw):
        WF.LAUNCH_COUNTS.clear()
        WF.categorical_nll(z, y, **kw).backward()
        out = dict(WF.LAUNCH_COUNTS)
        WF.LAUNCH_COUNTS.clear()
        return out

    assert launches() == {"whvi_categorical_nll_f32": 2, "whvi_categorical_nll_bwd_f32": 1}
    assert launches(label_smoothing=0.0, weight=None, ignore_index=None) == launches()
    ex = {"whvi_categorical_nll_ex_f32": 2, "whvi_categorical_nll_bwd_ex_f32": 1}
    for kw in (dict(weight=torch.ones(K, device=dev())), dict(label_smoothing=0.1), dict(ignore_index=-100)):
        assert launches(**kw) == ex, kw
    # unit weights, no smoothing and an ignore_index no label has: the plain call's values
    z.grad = None
    a = WF.categorical_nll(z, y)
    a.backward()
    g = z.grad.clone()
    z.grad = None
    b = WF.categorical_nll(z, y, torch.ones(K, device=dev()), 0.0, -100)
    b.backward()
    assert abs(a.item() - b.item()) <= 1e-6 * abs(a.item()) and rel_err(z.grad.cpu().numpy(), g.cpu().numpy()) <= 1e-6


# ------------------------------------------------------------------------------------------------------------------ networks
BF16_U = 2.0 ** -8


def _net(kind, seed=0, **opts):
    import whvi_b200 as W
    torch.manual_seed(seed)
    x_shape = None
    if kind == "stacked":
        mods, d_in, K = [W.WHVILinear(64, 128, bias=True), nn.ReLU(), W.WHVILinear(128, 10, bias=True)], 64, 10
    elif kind == "square":
        mods, d_in, K = [W.WHVILinear(256, 1024), nn.ReLU(), W.WHVILinear(1024, 1024, bias=True)], 256, 1024
    elif kind == "column":     # a Column layer (1 -> 64) in front of a Stacked head
        mods, d_in, K = [W.WHVILinear(1, 64, bias=True), nn.ReLU(), W.WHVILinear(64, 10, bias=True)], 1, 10
    elif kind == "linear":     # a foreign module as the head
        mods, d_in, K = [W.WHVILinear(64, 64, bias=True), nn.ReLU(), nn.Linear(64, 5)], 64, 5
    elif kind == "dense":
        mods, d_in, K = [W.WHVILinear(64, 128, covariance="dense"), nn.ReLU(), W.WHVILinear(128, 7, covariance="dense")], 64, 7
    elif kind == "cnn":
        mods = [W.WHVIConv2d(3, 8, 3, padding=1, lambda_=1.0, bias=True), nn.ReLU(), nn.Flatten(), W.WHVILinear(288, 10, bias=True)]
        d_in, K, x_shape = None, 10, (3, 6, 6)
    else:
        raise ValueError(kind)
    net = W.WHVIClassification(mods, train_samples=4, eval_samples=8, **opts).to(dev())
    with torch.no_grad():   # a posterior with visible noise, and O(1) logits
        for name, p in net.named_parameters():
            if name.endswith("g_mu"):
                p.normal_()
            elif kind == "cnn" and name.endswith(("s1", "s2")):
                p.normal_(0.0, p.numel() ** -0.5)
    return net, (x_shape if x_shape else (d_in,)), K


def _inject(net, S, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    for layer in net._whvi_layers():
        for blk in layer.square_blocks():
            blk.inject_eps(torch.randn((S, blk.D), device=dev(), generator=g))


def _options(K, seed):
    g = torch.Generator().manual_seed(seed)
    w = torch.rand(K, generator=g) * 2.0 + 0.1
    w[::3] = 0.0
    return dict(weight=w, label_smoothing=0.1, ignore_index=-100)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,bf16", [("stacked", False), ("square", False), ("column", False), ("linear", False), ("dense", False),
                                       ("cnn", False), ("stacked", True), ("square", True), ("cnn", True)])
def test_network_loss_and_gradients_match_torch_cross_entropy(kind, bf16):
    K0 = {"stacked": 10, "square": 1024, "column": 10, "linear": 5, "dense": 7, "cnn": 10}[kind]
    opts = _options(K0, 5)
    net, x_shape, K = _net(kind, **opts)
    S, B, n = net.train_samples, 48, 1000
    g = torch.Generator(device=dev()).manual_seed(1)
    x = torch.randn((B, *x_shape), device=dev(), generator=g)
    if kind == "square":
        x = x * 0.25   # logits of a few units: saturated bf16 logits move the softmax by far more than 2^-8
    if bf16:
        x = x.to(torch.bfloat16)
    y = torch.randint(0, K, (B,), device=dev(), generator=g)
    y[::5] = -100
    ref = copy.deepcopy(net)
    _inject(net, S, 7)
    loss = net.loss(x, y, n=n)
    loss.backward()
    _inject(ref, S, 7)
    logits = ref._run(x, S)
    assert logits.shape == (S, B, K)
    ce = F.cross_entropy(logits.double().reshape(S * B, K), y.repeat(S), weight=opts["weight"].double().to(dev()),
                         label_smoothing=0.1, ignore_index=-100, reduction="sum")
    ref_loss = (n / (B * S)) * ce + ref.kl
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) <= 1e-5 * abs(ref_loss.item())
    tol = 8 * BF16_U * len(net._whvi_layers()) if bf16 else 1e-5
    for (name, p), q in zip(net.named_parameters(), ref.parameters()):
        assert p.grad is not None and q.grad is not None, name
        assert rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) <= tol, name


def _blobs(n, seed):
    g = torch.Generator(device=dev()).manual_seed(seed)
    centres = torch.tensor([[2.0, 0.0], [-1.0, 1.7], [-1.0, -1.7]], device=dev())
    y = torch.randint(0, 3, (n,), device=dev(), generator=g)
    x = centres[y] + 0.5 * torch.randn((n, 2), device=dev(), generator=g)
    y[::7] = -100
    return torch.cat([x, torch.zeros((n, 14), device=dev())], 1), y


@pytest.mark.gpu
def test_cuda_graph_step_equals_eager_step():
    """Posterior noise off (softplus(-30) ~ 1e-13 next to O(1) means), so both runs see the same weights."""
    import whvi_b200 as W
    from whvi_b200 import FlatAdam, FlatParams
    from whvi_b200.graphs import GraphedTrainStep
    torch.manual_seed(0)
    eager = W.WHVIClassification([W.WHVILinear(16, 64, lambda_=1.0, bias=True), nn.ReLU(), W.WHVILinear(64, 3, lambda_=1.0, bias=True)],
                                 train_samples=2, eval_samples=16, weight=torch.tensor([1.0, 0.5, 2.0]), label_smoothing=0.1,
                                 ignore_index=-100).to(dev())
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
@pytest.mark.parametrize("kind", ["stacked", "cnn"])
def test_evaluation_over_the_labelled_rows(kind):
    """eval_model and predictive_metrics of a network with ignore_index (and weights and smoothing, which evaluation does not
    use) equal the plain network's metrics on the labelled subset, with the same noise."""
    K0 = 10
    net, x_shape, K = _net(kind, **_options(K0, 9))
    plain, _, _ = _net(kind)
    plain.load_state_dict(net.state_dict())
    net.eval()
    plain.eval()
    S, B = net.eval_samples, 300
    g = torch.Generator(device=dev()).manual_seed(2)
    x = torch.randn((B, *x_shape), device=dev(), generator=g)
    y = torch.randint(0, K, (B,), device=dev(), generator=g)
    y[::4] = -100
    keep = y != -100
    assert S <= 16   # one chunk: one injection gives each call the same noise, and a row's sums do not depend on the others
    _inject(net, S, 11)
    err, mnll = net.eval_model(x, y)
    _inject(plain, S, 11)
    err0, mnll0 = plain.eval_model(x[keep], y[keep])
    assert err == err0 and abs(mnll - mnll0) <= 1e-6 * abs(mnll0)
    _inject(net, S, 11)
    m = net.predictive_metrics(x, y)
    _inject(plain, S, 11)
    m0 = plain.predictive_metrics(x[keep], y[keep])
    assert m.keys() == m0.keys()
    for k in m:
        assert abs(m[k] - m0[k]) <= 1e-6 * max(abs(m0[k]), 1e-6), (k, m[k], m0[k])
    # a user loss gets every row of forward()'s logits; the MNLL is still the plain one over the labelled rows
    _inject(net, S, 11)
    seen = {}
    err2, mnll2 = net.eval_model(x, y, loss=lambda yp, yt: seen.setdefault("shape", tuple(yp.shape)) and 0.0)
    assert seen["shape"] == (B, K, S) and abs(mnll2 - mnll0) <= 1e-5 * abs(mnll0)


@pytest.mark.gpu
def test_training_step_with_options_adds_exactly_the_ex_launches():
    from whvi_b200 import functional as WF
    net, x_shape, K = _net("stacked", **_options(10, 3))
    x = torch.randn((16, *x_shape), device=dev())
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
    assert {k: v for k, v in extra.items() if v} == {"whvi_categorical_nll_ex_f32": 2, "whvi_categorical_nll_bwd_ex_f32": 1}
    assert math.isfinite(net.loss(x, y, n=100).item())
