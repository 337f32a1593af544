"""Predictive uncertainty of classifiers: the uncertainty instance of the sm_100a predictive kernel (``csrc/categorical.cu``,
``whvi_categorical_uncertainty_*``) up to ``WHVIClassification.predictive_uncertainty`` / ``predictive_metrics`` and
``distributed.reduce_predictive_uncertainty``; and ``WHVIRegression.predictive_uncertainty``.

CPU: an fp64 numpy restatement of the four sums tied to torch fp64, the new symbols, argument validation (shim and ctypes
alike), the front end's input checks, the Brier score and ECE against direct loops, the decomposition from the sums, and the
sample-sharded reduction in one process and across a gloo world of two.
GPU: the kernel against the restatement in every work-split regime, bit equality with the predictive call, chunking and bf16,
NaN labels, extreme logits, the networks against fp64 on their own logits, sample-sharded sums and launch accounting."""
import ctypes
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn

from conftest import rel_err

E_NULL, E_SHAPE, E_ALIGN, E_MODE = -1, -2, -3, -4
A = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference
NEW = ["whvi_categorical_uncertainty_f32", "whvi_categorical_uncertainty_bf16"]
# how far below zero fp32 rounding of the sums may take the mutual information, per unit of log K
MI_ROUNDING = 1e-5


# fp64 numpy restatement.  z: (S, B, K) logits, y: (B,) labels or None.  A class with p = 0 adds nothing to the entropy; a
# label outside [0, K) gives NaN in its input's log-likelihood sums.
def _lse(z):
    m = z.max(axis=-1, keepdims=True)
    m = np.where(np.isfinite(m), m, 0.0)
    return (m + np.log(np.exp(z - m).sum(axis=-1, keepdims=True)))[..., 0]


def ref_uncertainty(z, y=None):
    """(prob_sum (B, K), ent_sum (B,), loglik_sum (B,) or None, logpred (B,) or None) summed over s."""
    z = np.asarray(z, dtype=np.float64)
    lse = _lse(z)
    with np.errstate(invalid="ignore", divide="ignore"):
        p = np.exp(z - lse[..., None])
        ent = np.where(p > 0, p * (lse[..., None] - z), 0.0).sum(-1)
    prob = p.sum(0)
    if y is None:
        return prob, ent.sum(0), None, None
    y = np.asarray(y, dtype=np.int64)
    K = z.shape[-1]
    ok = (y >= 0) & (y < K)
    zy = np.take_along_axis(z, np.broadcast_to(np.where(ok, y, 0)[None, :, None], z.shape[:-1] + (1,)), axis=-1)[..., 0]
    lpy = np.where(ok[None, :], zy - lse, np.nan)
    return prob, ent.sum(0), lpy.sum(0), np.logaddexp.reduce(lpy, axis=0)


def _special_logits(rng, S, B, K):
    """Gaussian rows with rows of -inf logits, all-equal rows and one-hot-like (+-1e4) rows mixed in."""
    z = rng.standard_normal((S, B, K)) * 3.0
    z[:, 1::7, ::3] = -np.inf                      # masked classes (class 1 stays finite: label those rows 1)
    z[:, 2::7] = 0.5                               # all equal: entropy log K
    z[:, 3::7] = -1e4
    z[:, 3::7, 1] = 1e4                            # one-hot-like: entropy 0
    z[:, 4::7] = rng.uniform(-100.0, 100.0, size=z[:, 4::7].shape)
    return z


@pytest.mark.parametrize("K", [2, 3, 10, 33, 1000])
def test_restatement_equals_torch_fp64(K):
    rng = np.random.default_rng(K)
    S, B = 3, 41
    z = _special_logits(rng, S, B, K)
    y = rng.integers(0, K, size=B)
    y[1::7] = 1
    prob, ent, ll, lp = ref_uncertainty(z, y)
    zt = torch.from_numpy(z)
    yt = torch.from_numpy(y).reshape(1, B, 1).expand(S, B, 1)
    assert rel_err(prob, torch.softmax(zt, -1).sum(0).numpy()) <= 1e-12
    assert rel_err(ent, torch.distributions.Categorical(logits=zt).entropy().sum(0).numpy()) <= 1e-12
    logp = torch.log_softmax(zt, -1).gather(-1, yt)[..., 0]
    assert rel_err(ll, logp.sum(0).numpy()) <= 1e-12
    assert rel_err(lp, torch.logsumexp(logp, 0).numpy()) <= 1e-12
    h = ent / S
    assert np.allclose(h[2::7], math.log(K), rtol=1e-12) and np.all(h[3::7] == 0.0)
    assert np.all(h >= 0) and np.all(h <= math.log(K) * (1 + 1e-12))


def test_restatement_bad_labels_and_confident_wrong_rows():
    z = np.zeros((2, 3, 4))
    z[:, :, 0] = 200.0                             # p(y = 1) = e^-200 per sample: its log sum stays finite
    prob, ent, ll, lp = ref_uncertainty(z, np.array([1, -1, 4]))
    assert np.isnan(ll[1:]).all() and np.isnan(lp[1:]).all() and np.isfinite(prob).all() and np.isfinite(ent).all()
    assert abs(lp[0] - (math.log(2) - 200.0)) < 1e-9 and ll[0] == pytest.approx(-400.0)


def test_new_symbols_declared_exported_and_counted():
    from test_abi import declared_symbols
    from whvi_b200 import _lib
    from whvi_b200 import functional as WF
    L = ctypes.CDLL(str(_lib.LIB_PATH))
    declared = declared_symbols()
    for name in NEW:
        assert name in declared and hasattr(L, name) and name in _lib.SIGNATURES, name
        assert WF._LAUNCHES_PER_CALL[name] == 1, name


def _unc(**kw):
    a = dict(logits=A, stride=30, labels=A, prob=A, ll=A, lp=A, ent=A, S=2, B=3, K=10, flags=0, stream=None)
    a.update(kw)
    return tuple(a.values())


CASES = [
    (_unc(K=1), E_SHAPE, "outside [2, 65536]"),
    (_unc(K=65537), E_SHAPE, "outside [2, 65536]"),
    (_unc(S=-1), E_SHAPE, "S=-1"),
    (_unc(B=-3), E_SHAPE, "B=-3"),
    (_unc(flags=2), E_MODE, "unknown flags"),
    (_unc(stride=29), E_SHAPE, "sample_stride"),
    (_unc(S=1 << 40, stride=1 << 30), E_SHAPE, "too large"),
    (_unc(labels=None), E_NULL, "all be given"),
    (_unc(ll=None), E_NULL, "all be given"),
    (_unc(lp=None), E_NULL, "all be given"),
    (_unc(labels=None, ll=None), E_NULL, "all be given"),
    (_unc(prob=None), E_NULL, "null pointer"),
    (_unc(ent=None), E_NULL, "null pointer"),
    (_unc(logits=None), E_NULL, "null pointer"),
    (_unc(prob=A + 2), E_ALIGN, "aligned"),
    (_unc(labels=A + 4), E_ALIGN, "aligned"),
    (_unc(ll=A + 1), E_ALIGN, "aligned"),
    (_unc(lp=A + 2), E_ALIGN, "logpred and ent_sum"),
    (_unc(ent=A + 1), E_ALIGN, "logpred and ent_sum"),
]


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_validation_codes_and_messages_shim_equals_ctypes(dtype):
    from whvi_b200 import _lib
    L = _lib.lib()
    name = f"whvi_categorical_uncertainty_{dtype}"
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    fast = getattr(L, name)
    assert not hasattr(fast, "argtypes")          # all-integer call: handed out behind the shim
    for args, code, msg in CASES:
        rc_fast, msg_fast = fast(*args), L.whvi_last_error().decode()
        rc_raw, msg_raw = getattr(L._cdll, name)(*args), L.whvi_last_error().decode()
        assert rc_fast == rc_raw == code, (args, rc_fast, rc_raw, msg_fast)
        assert msg_fast == msg_raw and msg in msg_fast and name[5:] in msg_fast, msg_fast
    # bf16 logits need 2-byte alignment, fp32 logits 4: both fail at 1
    assert fast(*_unc(logits=A + 1)) == E_ALIGN
    # an empty batch is a valid no-op that needs no pointers (no launch); without labels only prob and ent are required
    assert fast(*_unc(logits=None, labels=None, ll=None, lp=None, prob=None, ent=None, B=0)) == 0
    # the predictive entry point keeps its own pairing rule and message
    pred = getattr(L, f"whvi_categorical_predictive_{dtype}")
    assert pred(A, 30, None, A, A, 2, 3, 10, 0, None) == E_NULL and "both be given" in L.whvi_last_error().decode()
    assert pred(A, 30, A, A, A, 2, 3, 10, 2, None) == E_MODE


def test_front_end_rejects_bad_inputs_without_fallback():
    from whvi_b200 import functional as WF
    z = torch.randn(2, 3, 4)
    y = torch.tensor([0, 1, 2])
    prob, v = torch.empty(3, 4), torch.empty(3)
    with pytest.raises(RuntimeError, match="CUDA"):
        WF.categorical_uncertainty_(z, None, prob, v)
    with pytest.raises(RuntimeError, match="CUDA"):
        WF.categorical_uncertainty_(z, y, prob, v, v.clone(), v.clone())
    with pytest.raises(RuntimeError, match="int64"):
        WF.categorical_uncertainty_(z, y.to(torch.int32), prob, v, v.clone(), v.clone())
    with pytest.raises(RuntimeError, match="labels must be"):
        WF.categorical_uncertainty_(z, torch.tensor([0]), prob, v, v.clone(), v.clone())
    with pytest.raises(RuntimeError, match=r"\(S, B, K\)"):
        WF.categorical_uncertainty_(z[0], None, prob, v)
    with pytest.raises(RuntimeError, match="float32 or bfloat16"):
        WF.categorical_uncertainty_(z.double(), None, prob, v)


def _np_ece(p, y, n_bins):
    conf, pred = p.max(1), p.argmax(1)
    total = 0.0
    for i in range(n_bins):
        lo, hi = i / n_bins, (i + 1) / n_bins
        sel = [b for b in range(len(y)) if (lo < conf[b] <= hi) or (i == 0 and conf[b] == 0.0)]
        if sel:
            acc = np.mean([pred[b] == y[b] for b in sel])
            total += len(sel) / len(y) * abs(acc - np.mean(conf[sel]))
    return total


@pytest.mark.parametrize("n_bins", [1, 10, 15])
def test_brier_and_ece_against_direct_numpy(n_bins):
    from whvi_b200.uncertainty import brier_score, expected_calibration_error
    rng = np.random.default_rng(n_bins)
    B, K = 500, 7
    p = rng.dirichlet(np.full(K, 0.3), size=B)
    p[:5] = np.eye(K)[:5]                           # confidence exactly 1 (last bin)
    p[5] = 1.0 / K
    y = rng.integers(0, K, size=B)
    brier = np.mean([sum((p[b, k] - (k == y[b])) ** 2 for k in range(K)) for b in range(B)])
    pt, yt = torch.from_numpy(p), torch.from_numpy(y)
    assert abs(brier_score(pt, yt) - brier) <= 1e-12
    assert abs(expected_calibration_error(pt, yt, n_bins) - _np_ece(p, y, n_bins)) <= 1e-12
    assert abs(expected_calibration_error(pt.float(), yt, n_bins) - expected_calibration_error(pt.float().double(), yt, n_bins)) == 0


def test_decomposition_from_sums():
    from whvi_b200.uncertainty import categorical_uncertainty
    rng = np.random.default_rng(0)
    S, B, K = 5, 30, 6
    z = _special_logits(rng, S, B, K)
    y = rng.integers(0, K, size=B)
    y[1::7] = 1
    prob, ent, _, lp = ref_uncertainty(z, y)
    u = categorical_uncertainty(torch.from_numpy(prob).float(), torch.from_numpy(ent).float(), torch.from_numpy(lp).float(), S)
    pbar = np.exp(z - _lse(z)[..., None]).mean(0)
    with np.errstate(divide="ignore", invalid="ignore"):
        h = -np.where(pbar > 0, pbar * np.log(pbar), 0.0).sum(1)
    assert u.S == S and u.probs.dtype == torch.float32 and u.predictive_entropy.dtype == torch.float64
    assert rel_err(u.predictive_entropy.numpy(), h) <= 1e-6 and rel_err(u.expected_entropy.numpy(), ent / S) <= 1e-6
    assert torch.equal(u.mutual_information, u.predictive_entropy - u.expected_entropy)
    assert (u.mutual_information.numpy() >= -MI_ROUNDING * math.log(K)).all()
    assert rel_err(u.log_predictive.numpy(), lp - math.log(S)) <= 1e-6
    assert categorical_uncertainty(torch.from_numpy(prob), torch.from_numpy(ent), None, S).log_predictive is None
    with pytest.raises(ValueError):
        categorical_uncertainty(torch.from_numpy(prob), torch.from_numpy(ent), None, 0)


def _shard_sums(z, y, s0, s1):
    prob, ent, ll, lp = ref_uncertainty(z[s0:s1], y)
    return [torch.from_numpy(a).float() for a in (prob, ent, lp, ll)]


def _sharded_case():
    rng = np.random.default_rng(7)
    S, B, K = 6, 9, 5
    z = rng.standard_normal((S, B, K)) * 3
    y = rng.integers(0, K, size=B)
    z[:, 2, :] = -1e4
    z[:, 2, 0] = 1e4                                # label 0 wins: finite
    z[:, 3, :] = 0.0
    z[:, 3, 1] = 200.0                              # y = 0 while class 1 has p ~ 1: log p(y) ~ -200, exp underflows in fp32
    y[2], y[3] = 0, 0
    y[5] = -1                                       # NaN row
    return S, z, y


def test_reduce_predictive_uncertainty_single_process():
    from whvi_b200.distributed import reduce_predictive_uncertainty
    from whvi_b200.uncertainty import categorical_uncertainty
    S, z, y = _sharded_case()
    prob, ent, lp, ll = _shard_sums(z, y, 0, S)
    u, mean_ll = reduce_predictive_uncertainty(prob.clone(), ent.clone(), lp.clone(), ll.clone(), S)
    ref = categorical_uncertainty(prob, ent, lp, S)
    for a, b in zip(u[:5], ref[:5]):
        assert torch.equal(a.isnan(), b.isnan()) and torch.allclose(a[~a.isnan()], b[~b.isnan()].to(a.dtype), rtol=1e-6, atol=0)
    assert torch.isnan(u.log_predictive[5]) and torch.isfinite(u.log_predictive[3]) and u.log_predictive[3] < -150
    assert torch.allclose(mean_ll[~mean_ll.isnan()], (ll / S)[~mean_ll.isnan()])
    u2, none = reduce_predictive_uncertainty(prob.clone(), ent.clone(), None, None, S)
    assert none is None and u2.log_predictive is None


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from whvi_b200.distributed import reduce_predictive_uncertainty, shard_samples
        S, z, y = _sharded_case()
        first, n_local = shard_samples(S, rank, world)
        prob, ent, lp, ll = _shard_sums(z, y, first, first + n_local)
        if rank == 1:
            lp[4] = float("-inf")                   # -inf on one rank only: the other rank's value survives
        u, mean_ll = reduce_predictive_uncertainty(prob, ent, lp, ll, n_local)
        rprob, rent, rll, rlp = ref_uncertainty(z, y)
        n0 = shard_samples(S, 0, world)[1]
        rlp[4] = ref_uncertainty(z[:n0], y)[3][4]   # rank 0's samples alone
        got, want = u.log_predictive.numpy(), rlp - math.log(S)
        rest = [b for b in range(len(y)) if b != 5]
        ok = u.S == S and rel_err(u.probs.numpy(), rprob / S) <= 1e-6 and rel_err(u.expected_entropy.numpy(), rent / S) <= 1e-6
        ok = ok and bool(np.isnan(got[5])) and not np.isnan(got[rest]).any() and float(np.max(np.abs(got[rest] - want[rest]))) <= 1e-5
        ok = ok and got[3] < -150 and bool(np.isnan(mean_ll[5].item())) and rel_err(mean_ll.numpy()[rest], rll[rest] / S) <= 1e-6
        # all ranks -inf: stays -inf (no NaN from -inf - -inf)
        u3, _ = reduce_predictive_uncertainty(prob, ent, torch.full_like(lp, float("-inf")), ll, n_local)
        ok = ok and bool(torch.all(u3.log_predictive == float("-inf")))
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_reduce_predictive_uncertainty_gloo_two_ranks():
    world = 2
    port = _free_port()
    ctx = mp.get_context("spawn")
    out = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert all(out.get(r) for r in range(world)), dict(out)


def test_regression_uncertainty_without_fused_sums():
    import whvi_b200 as W
    torch.manual_seed(0)
    net = W.WHVIRegression([nn.Linear(3, 2)], sigma=0.5)
    u = net.predictive_uncertainty(torch.randn(4, 3), n_samples=5)
    assert u.S == 5 and u.mean.shape == (4, 2) and u.mean.dtype == torch.float64
    assert torch.all(u.epistemic_variance == 0) and torch.allclose(u.aleatoric_variance, torch.full((4, 2), 0.25, dtype=torch.float64))


# ------------------------------------------------------------------------------------------------------------------ GPU
def dev():
    return torch.device("cuda:0")


def _call(zt, yt, S=None, stride=None, flags=0, fill=float("nan"), outs=None):
    """The uncertainty entry point on device tensors, every output prefilled (NaN by default); returns (prob, ent, ll, lp)."""
    from whvi_b200 import _lib
    S = zt.shape[0] if S is None else S
    B, K = zt.shape[1], zt.shape[2]
    sfx = "bf16" if zt.dtype == torch.bfloat16 else "f32"
    if outs is None:
        outs = (torch.full((B, K), fill, device=dev()), torch.full((B,), fill, device=dev()),
                torch.full((B,), fill, device=dev()), torch.full((B,), fill, device=dev()))
    prob, ent, ll, lp = outs
    lab = yt is not None
    name = f"whvi_categorical_uncertainty_{sfx}"
    rc = getattr(_lib.lib(), name)(zt.data_ptr(), B * K if stride is None else stride, yt.data_ptr() if lab else None, prob.data_ptr(),
                                   ll.data_ptr() if lab else None, lp.data_ptr() if lab else None, ent.data_ptr(), S, B, K, flags,
                                   torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, name)
    return outs


def _pred(zt, yt):
    from whvi_b200 import _lib
    S, B, K = zt.shape
    prob, ll = torch.full((B, K), float("nan"), device=dev()), torch.full((B,), float("nan"), device=dev())
    name = "whvi_categorical_predictive_bf16" if zt.dtype == torch.bfloat16 else "whvi_categorical_predictive_f32"
    _lib.check(getattr(_lib.lib(), name)(zt.data_ptr(), B * K, yt.data_ptr(), prob.data_ptr(), ll.data_ptr(), S, B, K, 0,
                                         torch.cuda.current_stream().cuda_stream), name)
    return prob, ll


def _check_against_ref(got, z, y, tol=1e-5):
    prob, ent, ll, lp = (t.cpu().numpy() for t in got)
    rprob, rent, rll, rlp = ref_uncertainty(z, y)
    assert rel_err(prob, rprob) <= tol
    assert rel_err(ent, rent) <= tol
    if y is not None:
        assert rel_err(ll, rll) <= tol and rel_err(lp, rlp) <= tol


# inputs B per call (the predictive plans on B): 256 / TPR inputs per CTA pass, 148 * 16 CTAs before the grid strides.  B gives
# a partial last group and, for K = 2 ... 1000 and K = 4096, more inputs than one pass of the capped grid
ROWS = {2: 303333, 3: 151653, 10: 38002, 17: 19002, 33: 19002, 100: 19002, 1000: 19002, 2048: 2402, 2049: 2402, 4096: 2402,
        65536: 1202}


@pytest.mark.gpu
@pytest.mark.parametrize("K", sorted(ROWS))
def test_kernel_against_fp64_restatement(K):
    S, B = 3, ROWS[K]
    g = torch.Generator(device=dev()).manual_seed(K)
    zt = torch.randn((S, B, K), device=dev(), generator=g) * 3
    zt[:, 1::5] = (torch.rand((S, (B + 3) // 5, K), device=dev(), generator=g)[:, :zt[:, 1::5].shape[1]] - 0.5) * 200
    yt = torch.randint(0, K, (B,), device=dev(), generator=g)
    z, y = zt.cpu().numpy(), yt.cpu().numpy()
    got = _call(zt, yt)
    _check_against_ref(got, z, y)
    # prob_sum and loglik_sum are the predictive call's bits
    prob, ll = _pred(zt, yt)
    assert torch.equal(got[0], prob) and torch.equal(got[2], ll)
    # bit-reproducible, independent of what the buffers held
    for a, b in zip(got, _call(zt, yt, fill=0.0)):
        assert torch.equal(a, b)
    # without labels: the same prob_sum and ent_sum
    nolab = _call(zt, None)
    assert torch.equal(nolab[0], got[0]) and torch.equal(nolab[1], got[1])
    # sample chunks (strided slices of the same tensor) continued with ACCUMULATE equal one call
    outs = tuple(torch.full_like(t, float("nan")) for t in got)
    for s0, s1 in ((0, 1), (1, S)):
        _call(zt[s0:s1], yt, flags=1 if s0 else 0, outs=outs)
    for a, b in zip(outs, got):
        assert torch.equal(a, b)
    # bf16: the fp32 instance on the widened logits, bit for bit
    zb = zt.to(torch.bfloat16)
    for a, b in zip(_call(zb, yt), _call(zb.float(), yt)):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 1000, 4096])
def test_sample_stride_and_empty_sample_sets(K):
    S, B = 4, 37
    g = torch.Generator(device=dev()).manual_seed(1)
    big = torch.randn((S, B + 5, K), device=dev(), generator=g) * 3   # sample stride (B + 5) K > B K
    yt = torch.randint(0, K, (B,), device=dev(), generator=g)
    zt = big[:, :B]
    got = _call(zt, yt, stride=(B + 5) * K)
    _check_against_ref(got, zt.cpu().numpy(), yt.cpu().numpy())
    for a, b in zip(got, _call(zt.contiguous(), yt)):
        assert torch.equal(a, b)
    # S = 0 without ACCUMULATE: zero sums and logpred = log 0 = -inf; with ACCUMULATE: nothing changes
    prob, ent, ll, lp = _call(zt, yt, S=0)
    assert torch.all(prob == 0) and torch.all(ent == 0) and torch.all(ll == 0) and torch.all(lp == float("-inf"))
    keep = tuple(t.clone() for t in got)
    _call(zt, yt, S=0, flags=1, outs=got)
    for a, b in zip(got, keep):
        assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [10, 1000, 4096])
def test_labels_outside_range_give_nan_in_label_sums_only(K):
    S, B = 3, 37
    g = torch.Generator(device=dev()).manual_seed(3)
    zt = torch.randn((S, B, K), device=dev(), generator=g) * 3
    y = torch.randint(0, K, (B,), device=dev(), generator=g)
    bad = y.clone()
    bad[5], bad[20] = -1, K
    p0, e0, ll0, lp0 = _call(zt, y)
    p1, e1, ll1, lp1 = _call(zt, bad)
    keep = [b for b in range(B) if b not in (5, 20)]
    assert torch.equal(p0, p1) and torch.equal(e0, e1)
    assert torch.isnan(ll1[[5, 20]]).all() and torch.isnan(lp1[[5, 20]]).all()
    assert torch.equal(ll1[keep], ll0[keep]) and torch.equal(lp1[keep], lp0[keep])


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 10, 33, 1000, 4096])
def test_extreme_logits(K):
    from whvi_b200.uncertainty import categorical_uncertainty
    S, B = 5, 700
    rng = np.random.default_rng(K)
    z = _special_logits(rng, S, B, K).astype(np.float32)
    z[:, 5::7] = z[0, 5::7][None]                    # the samples agree: mutual information 0 up to rounding
    y = rng.integers(0, K, size=B)
    y[1::7] = 1
    y[3::7] = 0                                      # one-hot-like rows with the wrong label: log p = -2e4, finite
    zt, yt = torch.from_numpy(z).to(dev()), torch.from_numpy(y).to(dev())
    got = _call(zt, yt)
    prob, ent, ll, lp = got
    for t in got:
        assert not torch.isnan(t).any()
    _check_against_ref(got, z, y)
    h = ent / S
    assert torch.all(h >= 0) and torch.all(h <= math.log(K) * (1 + 1e-6))
    u = categorical_uncertainty(prob, ent, lp, S)
    assert torch.all(u.mutual_information >= -MI_ROUNDING * math.log(K))
    assert torch.all(torch.isfinite(u.log_predictive)) and torch.all(u.log_predictive[3::7] < -1e4)
    assert torch.all(u.mutual_information[5::7].abs() <= MI_ROUNDING * math.log(K))


# ------------------------------------------------------------------------------------------------------------------ networks
def _net(kind, seed=0):
    import whvi_b200 as W
    torch.manual_seed(seed)
    x_shape = None
    if kind == "stacked":
        mods, d_in, K = [W.WHVILinear(64, 128, bias=True), nn.ReLU(), W.WHVILinear(128, 10, bias=True)], 64, 10
    elif kind == "square":
        mods, d_in, K = [W.WHVILinear(256, 1024), nn.ReLU(), W.WHVILinear(1024, 1024, bias=True)], 256, 1024
    elif kind == "linear":
        mods, d_in, K = [W.WHVILinear(64, 64, bias=True), nn.ReLU(), nn.Linear(64, 5)], 64, 5
    elif kind == "dense":
        mods, d_in, K = [W.WHVILinear(64, 128, covariance="dense"), nn.ReLU(), W.WHVILinear(128, 7, covariance="dense")], 64, 7
    elif kind == "cnn":
        mods = [W.WHVIConv2d(3, 8, 3, padding=1, lambda_=1.0, bias=True), nn.ReLU(), nn.Flatten(), W.WHVILinear(288, 10, bias=True)]
        d_in, K, x_shape = None, 10, (3, 6, 6)
    else:
        raise ValueError(kind)
    net = W.WHVIClassification(mods, train_samples=4, eval_samples=8).to(dev())
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


@pytest.mark.gpu
@pytest.mark.parametrize("kind,bf16", [("stacked", False), ("square", False), ("linear", False), ("dense", False), ("cnn", False),
                                       ("stacked", True), ("square", True), ("cnn", True)])
def test_predictive_uncertainty_equals_fp64_from_logits(kind, bf16):
    net, x_shape, K = _net(kind)
    net.eval()
    S, B = net.eval_samples, 300
    g = torch.Generator(device=dev()).manual_seed(2)
    x = torch.randn((B, *x_shape), device=dev(), generator=g)
    if bf16:
        x = x.to(torch.bfloat16)
    y = torch.randint(0, K, (B,), device=dev(), generator=g)
    assert S <= 16   # one chunk, so one injection gives the call the noise of _run below
    _inject(net, S, 11)
    with torch.no_grad():
        logits = net._run(x, S).double()                            # (S, B, K)
    lp = torch.log_softmax(logits, -1)
    p = lp.exp()
    pbar = p.mean(0)
    ref_h = -torch.special.xlogy(pbar, pbar).sum(-1)
    ref_eh = -(torch.special.xlogy(p, p)).sum(-1).mean(0)
    ref_lpred = torch.logsumexp(lp.gather(-1, y.reshape(1, B, 1).expand(S, B, 1))[..., 0], 0) - math.log(S)
    _inject(net, S, 11)
    u = net.predictive_uncertainty(x, y)
    assert u.S == S and u.probs.shape == (B, K) and u.log_predictive.shape == (B,)
    assert rel_err(u.probs.cpu().numpy(), pbar.cpu().numpy()) <= 1e-5
    assert rel_err(u.predictive_entropy.cpu().numpy(), ref_h.cpu().numpy()) <= 1e-5
    assert rel_err(u.expected_entropy.cpu().numpy(), ref_eh.cpu().numpy()) <= 1e-5
    assert rel_err(u.log_predictive.cpu().numpy(), ref_lpred.cpu().numpy()) <= 1e-5
    mi_ref = (ref_h - ref_eh).cpu().numpy()
    assert np.max(np.abs(u.mutual_information.cpu().numpy() - mi_ref)) <= 1e-5 * max(math.log(K), 1.0)
    # probs are predict_proba's, bit for bit
    _inject(net, S, 11)
    assert torch.equal(u.probs, net.predict_proba(x))
    # the metrics from the same sums
    _inject(net, S, 11)
    m = net.predictive_metrics(x, y)
    err = float((pbar.argmax(1) != y).double().mean())
    mnll = float(-lp.gather(-1, y.reshape(1, B, 1).expand(S, B, 1)).sum() / S)
    assert m["error"] == err and abs(m["nll"] + float(ref_lpred.mean())) <= 1e-5 * abs(float(ref_lpred.mean()))
    assert abs(m["mnll"] - mnll) <= 1e-5 * abs(mnll)
    onehot = torch.nn.functional.one_hot(y, K).double()
    assert abs(m["brier"] - float((pbar - onehot).square().sum(1).mean())) <= 1e-5
    assert 0.0 <= m["ece"] <= 1.0
    # without labels
    _inject(net, S, 11)
    u0 = net.predictive_uncertainty(x)
    assert u0.log_predictive is None and torch.equal(u0.expected_entropy, u.expected_entropy)


@pytest.mark.gpu
def test_chunked_uncertainty_equals_one_call_and_half_sample_shards_combine():
    from whvi_b200 import functional as WF
    from whvi_b200.uncertainty import categorical_uncertainty
    net, x_shape, K = _net("stacked")
    net.eval()
    S, B, chunk = 8, 50, 3
    x = torch.randn((B, *x_shape), device=dev())
    y = torch.randint(0, K, (B,), device=dev())
    chunks = [(s0, min(S, s0 + chunk)) for s0 in range(0, S, chunk)]
    for i, (s0, s1) in enumerate(chunks):
        _inject(net, s1 - s0, 100 + i)
    sums = net.predictive_uncertainty_sums(x, y, n_samples=S, chunk_samples=chunk)
    logits = []
    for i, (s0, s1) in enumerate(chunks):
        _inject(net, s1 - s0, 100 + i)
        with torch.no_grad():
            logits.append(net._run(x, s1 - s0))
    z = torch.cat(logits)
    whole = [torch.empty((B, K), device=dev())] + [torch.empty(B, device=dev()) for _ in range(3)]
    WF.categorical_uncertainty_(z, y, *whole)
    for a, b in zip(sums[:4], whole):
        assert torch.equal(a, b)
    # two "ranks" with half the samples each, combined as reduce_predictive_uncertainty does across ranks
    halves = []
    for s0, s1 in ((0, S // 2), (S // 2, S)):
        h = [torch.empty((B, K), device=dev())] + [torch.empty(B, device=dev()) for _ in range(3)]
        WF.categorical_uncertainty_(z[s0:s1], y, *h)
        halves.append(h)
    (p0, e0, l0, lp0), (p1, e1, l1, lp1) = halves
    u = categorical_uncertainty(p0 + p1, e0 + e1, torch.logaddexp(lp0.double(), lp1.double()), S)
    ref = categorical_uncertainty(*whole[:2], whole[3], S)
    for a, b in zip(u[:5], ref[:5]):
        assert torch.allclose(a.double(), b.double(), rtol=1e-5, atol=1e-6)
    assert torch.allclose(l0 + l1, whole[2], rtol=1e-5)


@pytest.mark.gpu
def test_predictive_uncertainty_launches_equal_predict_proba():
    from whvi_b200 import functional as WF
    net, x_shape, K = _net("stacked")
    net.eval()
    x = torch.randn((40, *x_shape), device=dev())
    y = torch.randint(0, K, (40,), device=dev())

    def count(fn):
        WF.LAUNCH_COUNTS.clear()
        fn()
        out = dict(WF.LAUNCH_COUNTS)
        WF.LAUNCH_COUNTS.clear()
        return out

    base = count(lambda: net.predict_proba(x, n_samples=20, chunk_samples=6))
    unc = count(lambda: net.predictive_uncertainty(x, y, n_samples=20, chunk_samples=6))
    assert base.pop("whvi_categorical_predictive_f32") == 4 and unc.pop("whvi_categorical_uncertainty_f32") == 4
    assert base == unc


@pytest.mark.gpu
def test_regression_uncertainty_fused_sums_and_fallback():
    import whvi_b200 as W
    torch.manual_seed(0)
    net = W.WHVIRegression([W.WHVILinear(64, 128, bias=True), nn.ReLU(), W.WHVILinear(128, 128, bias=True)], sigma=0.3,
                           eval_samples=8).to(dev())
    net.eval()
    x = torch.randn((20, 64), device=dev())
    assert net.predictive_sums(x) is not None      # ends in a square layer: the fused moments path
    _inject(net, 8, 5)
    u = net.predictive_uncertainty(x)
    _inject(net, 8, 5)
    with torch.no_grad():
        yh = net._run(x, 8).double()
    assert u.S == 8 and rel_err(u.mean.cpu().numpy(), yh.mean(0).cpu().numpy()) <= 1e-5
    assert rel_err(u.epistemic_variance.cpu().numpy(), yh.var(0, unbiased=False).cpu().numpy()) <= 1e-4
    assert torch.allclose(u.aleatoric_variance, torch.full_like(u.mean, 0.09), rtol=1e-6)
