"""The layer kernels against the fp64 oracle in every work-split regime they run in.

The persistent layer kernels cut the (S, B*D) activations into tiles, the tiles of a sample into CTAs, and the CTAs into
waves and workspace slabs; the backward then adds the slabs up in a fixed order (layer_bwd.cu, launch_bwd_reduce).  This
file restates that host-side plan in Python, pins the restatement to the library's own size queries (CPU), picks shapes
that reach each regime and checks on the CPU that every (kernel family, D, regime) cell has one, then runs the kernels at
those shapes against the fp64 oracle with the cached workspace poisoned (GPU), so a tile, slab or reduction step that a
kernel skips or adds twice shows up as NaN or as a large error.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import pytest
import torch

from conftest import rel_err

TOL = 1e-4
SMS = 148


# ------------------------------------------------------------------------------------------------- plan.cuh, restated
def _cdiv(a, b):
    return -(-a // b)


def make_plan(S, tiles_per_sample, groups, target_ctas, min_iters):
    """whvi::make_plan (plan.cuh:15-25)."""
    max_ctas = _cdiv(tiles_per_sample, groups)
    ctas = _cdiv(target_ctas, S)
    ctas = max(min(ctas, max_ctas), 1)
    iters = max(_cdiv(tiles_per_sample, ctas * groups), min_iters)
    ctas = _cdiv(tiles_per_sample, iters * groups)
    return ctas, iters


def make_plan_waves(S, tiles_per_sample, groups, slots, min_iters, max_waves):
    """whvi::make_plan_waves (plan.cuh:32-46)."""
    max_cps = max(_cdiv(tiles_per_sample, min_iters * groups), 1)
    best_cps, best_iters, best_cost = 1, _cdiv(tiles_per_sample, groups), -1
    cps = 1
    while cps <= max_cps and cps * S <= slots * max_waves:
        iters = _cdiv(tiles_per_sample, cps * groups)
        eff = _cdiv(tiles_per_sample, iters * groups)
        waves = _cdiv(eff * S, slots)
        cost = waves * iters
        if best_cost < 0 or cost < best_cost:
            best_cost, best_cps, best_iters = cost, eff, iters
        cps += 1
    return best_cps, best_iters


# ------------------------------------------------------------------------------------------------- launch tables
# Each entry: k = log2 D -> (tile bits N, groups or pairs per CTA, extra).
# Forward, launch_layer_fwd (layer_fwd.cu:256-282): extra = min_iters of make_plan(S, tiles, GROUPS, 148 * 16, min_iters),
# 4 for the two-view kernels (ROUNDS == 2), 2 for the three-view ones (layer_fwd.cu:221).
FWD = {**{k: (10, 4, 2) for k in range(2, 7)},     # three views
       **{k: (10, 8, 4) for k in range(7, 11)},    # two views, one warp per 1024-float tile
       11: (12, 2, 4), 12: (12, 2, 4),             # two views, 64 floats per thread
       13: (13, 1, 2), 14: (14, 1, 2), 15: (15, 1, 2)}
FWD_TARGET_CTAS = SMS * 16

# Backward, launch_layer_bwd (layer_bwd.cu:1131-1157), the tensor-memory kernels of the default build:
# layer_bwd_tma_kernel N = 10 with 4 pairs for k <= 10; layer_bwd_tm_kernel with N = 12 and 128 / 64 = 2 pairs for
# k = 11, 12, and N = 13 with 128 / 128 = 1 pair for k = 13 (launch_bwd_tm_cfg: PAIRS = 128 / T, T = 2^(N - 6)).
# Both plan with make_plan_waves(S, tiles, PAIRS, 148, 8, 8) (layer_bwd.cu:1044, 1093).  extra = None.
BWD = {**{k: (10, 4, None) for k in range(2, 11)}, 11: (12, 2, None), 12: (12, 2, None), 13: (13, 1, None)}

# Loss layer, launch_layer_loss (layer_loss.cu:379-406) and launch_layer_loss_tm (layer_loss_tm.cu:390-396): extra = the
# squared-error partials per slab, T / 32 with T = 2^(N - C) threads per role.  layer_loss.cu runs for k = 7..10 always and
# for k = 11, 12 with a bias; without a bias k = 11, 12 run the tensor-memory kernel.  Both plan with make_plan_waves(S,
# tiles, PAIRS, 148, 8, 8) (layer_loss.cu:352, layer_loss_tm.cu:367).
LOSS = {**{k: (10, 4, 1) for k in range(7, 11)},  # N = 10, C = 5: 32 threads per role
        11: (11, 2, 2), 12: (12, 1, 4)}          # N = 11 / 12, C = 5
LOSS_TM = {11: (12, 2, 2), 12: (12, 2, 2)}       # N = 12, C = 6

# Moments, launch_moments_cfg (layer_moments.cu:182-197): one row per tile, grid = min(tiles, (148 - reserve_sms) *
# ctas_per_sm), ctas_per_sm = 512 tensor-memory columns / (128 per thread * T / 128 warps), T = 2^(k - 6).
# The library has no size query that exposes this grid: the restatement is pinned by the comment only.
MOMENTS_CTAS_PER_SM = {13: 4, 14: 2, 15: 1}


def _log2(D):
    k = D.bit_length() - 1
    assert D == 1 << k
    return k


@dataclass(frozen=True)
class Split:
    """One launch's work split.  groups: tile groups (forward) or tile pairs (backward, loss) per CTA."""
    tile: int
    groups: int
    tiles: int        # tiles per sample
    cps: int          # CTAs per sample
    iters: int        # tiles per group (pair) per CTA
    grid: int         # CTAs of the launch

    @property
    def slabs(self):  # workspace slabs per sample (backward, loss)
        return self.cps * self.groups

    @property
    def last(self):   # tiles of a sample's last CTA (tile t goes to CTA t // (iters * groups), group t % groups)
        return self.tiles - (self.cps - 1) * self.iters * self.groups


def _split(S, B, D, N, groups, planner):
    tile = 1 << N
    tiles = _cdiv(B * D, tile)
    cps, iters = planner(S, tiles, groups)
    return Split(tile, groups, tiles, cps, iters, cps * S)


def fwd_split(S, B, D):
    N, groups, min_iters = FWD[_log2(D)]
    return _split(S, B, D, N, groups, lambda s, t, g: make_plan(s, t, g, FWD_TARGET_CTAS, min_iters))


def bwd_split(S, B, D):
    N, pairs, _ = BWD[_log2(D)]
    return _split(S, B, D, N, pairs, lambda s, t, g: make_plan_waves(s, t, g, SMS, 8, 8))


def loss_split(S, B, D, tm):
    N, pairs, _ = (LOSS_TM if tm else LOSS)[_log2(D)]
    return _split(S, B, D, N, pairs, lambda s, t, g: make_plan_waves(s, t, g, SMS, 8, 8))


def bwd_workspace_bytes(S, B, D):
    sp = bwd_split(S, B, D)
    return 4 * S * sp.cps * sp.groups * 4 * sp.tile


def loss_sizes(S, B, D):
    """(workspace bytes, squared-error partials) as whvi_layer_loss_sizes reports them: the larger of the two kernels at
    k = 11, 12, where the query cannot know whether the call will have a bias (layer_loss.cu:383-398)."""
    k = _log2(D)
    out = []
    for tm in ([False, True] if k in LOSS_TM else [False]):
        sp = loss_split(S, B, D, tm)
        T = 1 << ((12 - 6) if tm else (LOSS[k][0] - 5))
        assert T // 32 == (LOSS_TM if tm else LOSS)[k][2]
        out.append((4 * S * sp.slabs * 4 * sp.tile, S * sp.slabs * (T // 32)))
    return max(o[0] for o in out), max(o[1] for o in out)


def stacked_bwd_workspace_bytes(S, B, D, G, want_dx):
    """whvi_stacked_bwd_workspace_bytes (api.cu:538-567): dy blocks, [dx blocks], dg, 256-byte aligned, then the grouped
    layer backward's workspace for S * G virtual samples."""
    blocks = 4 * G * S * B * D
    o = blocks + (blocks if want_dx else 0) + 4 * G * S * D
    o = _cdiv(o, 256) * 256
    return o + bwd_workspace_bytes(S * G, B, D)


def moments_grid(B, D, reserve_sms=0):
    sms = SMS - (reserve_sms if 0 < reserve_sms < SMS else 0)
    return min(B, sms * MOMENTS_CTAS_PER_SM[_log2(D)])


def reduce_branches(S, sp, D, groups=1):
    """launch_bwd_reduce (layer_bwd.cu:1010-1028): (pass A runs, pass A's grid z, pass B's CTA-per-output branch)."""
    direct = D == sp.tile
    return sp.slabs > 1 or direct, min(S, 65535), (S // groups) * (sp.tile // D) >= 1024


# ------------------------------------------------------------------------------------------------- regimes
# R1  one CTA per sample, partial last tile (D < tile, B*D not a multiple of the tile)
# R2  several CTAs per sample; in the last CTA some tile groups or pairs get no tile at all (with one group per CTA: the
#     group runs out of tiles before its last iteration); for D < tile the last tile is partial
# R3  more CTAs than one wave of 148 (one-CTA-per-SM kernels: backward, loss)
# R4  >= 9 slabs per sample with (slabs - 1) % 4 != 0: pass A runs its 4-way loop and its remainder loop
# R5  pass B's CTA-per-output branch
# R6  S > 65535: pass A loops over grid z
# M1  moments: B > grid and B % grid != 0 (a CTA takes a second row and a row remains for part of the grid)
def _r1(sp, B, D):
    return sp.cps == 1 and D < sp.tile and (B * D) % sp.tile != 0


def _r2(sp, B, D):
    idle = sp.last < sp.groups if sp.groups > 1 else sp.last < sp.iters
    return sp.cps >= 2 and idle and (D >= sp.tile or (B * D) % sp.tile != 0)


def _r4(sp):
    return sp.slabs >= 9 and (sp.slabs - 1) % 4 != 0


def fwd_regimes(S, B, D):
    sp = fwd_split(S, B, D)
    return {r for r, ok in (("R1", _r1(sp, B, D)), ("R2", _r2(sp, B, D))) if ok}


def bwd_regimes(S, B, D, groups=1):
    """groups > 1: the grouped (Stacked) launch, S = G * samples virtual samples."""
    sp = bwd_split(S, B, D)
    _, _, cta_per_output = reduce_branches(S, sp, D, groups)
    return {r for r, ok in (("R1", _r1(sp, B, D)), ("R2", _r2(sp, B, D)), ("R3", sp.grid > SMS), ("R4", _r4(sp)),
                            ("R5", cta_per_output), ("R6", S > 65535)) if ok}


def loss_regimes(S, B, D, tm):
    sp = loss_split(S, B, D, tm)
    _, _, cta_per_output = reduce_branches(S, sp, D)
    return {r for r, ok in (("R1", _r1(sp, B, D)), ("R2", _r2(sp, B, D)), ("R3", sp.grid > SMS), ("R4", _r4(sp)),
                            ("R5", cta_per_output)) if ok}


def moments_regimes(B, D, reserve_sms=0):
    grid = moments_grid(B, D, reserve_sms)
    return {"M1"} if B > grid and B % grid != 0 else set()


# ------------------------------------------------------------------------------------------------- the shapes
# Chosen with the restated plan; test_every_regime_cell_is_covered says which cells each list must reach.  S >= 2 where
# it is cheap, so per-sample and shared inputs differ and the sample-minor CTA order is exercised.
FWD_SHAPES = ([(3, 7, D) for D in (4, 8, 16, 32, 64, 128, 256, 512, 2048)] +                           # R1
              [(2, 2049, 4), (2, 1025, 8), (2, 513, 16), (2, 257, 32), (2, 129, 64), (2, 257, 128),     # R2
               (2, 129, 256), (2, 65, 512), (2, 33, 1024), (2, 17, 2048), (2, 9, 4096), (2, 3, 8192),
               (2, 3, 16384), (2, 3, 32768)])
BWD_SHAPES = ([(149, 3, D) for D in (4, 8, 16, 32, 64, 128)] + [(256, 3, 256), (512, 3, 512), (512, 3, 2048)] +  # R1 R3 R5
              [(1024, 1, 1024), (1024, 1, 4096), (1024, 1, 8192)] +                                          # R3 R5
              [(2, 65537, 4), (2, 32769, 8), (2, 16385, 16), (2, 8193, 32), (2, 4097, 64), (2, 1793, 128),   # R2 R4
               (2, 897, 256), (2, 449, 512), (2, 227, 1024), (2, 225, 2048), (2, 113, 4096), (2, 73, 8192)])
R6_SHAPE = (65539, 1, 4)   # ~4.3 GB of workspace
# (S, B, D, bias): at D = 2048, 4096 a bias selects layer_loss.cu, no bias the tensor-memory kernel
LOSS_SHAPES = ([(149, 3, 128, True), (256, 3, 256, False), (512, 3, 512, True), (512, 3, 2048, False)] +        # R1 R3 R5
               [(1024, 1, 1024, False), (1024, 1, 2048, True), (1024, 1, 4096, True), (1024, 1, 4096, False)] +  # R3 R5
               [(2, 1793, 128, False), (2, 897, 256, True), (2, 449, 512, False), (2, 227, 1024, True),          # R2 R4
                (2, 113, 2048, True), (2, 225, 2048, False), (2, 73, 4096, True), (2, 113, 4096, False)] +
               [(149, 9, 2048, True), (149, 9, 4096, False)])                                                  # R3
# (n_in, n_out, S, B) of grouped Stacked calls: D = next_pow2(n_in), G = ceil(n_out / D); ragged n_in and n_out
STACKED_SHAPES = [(998, 1499, 2, 227),   # G = 2 at D = 1024: R2 R4
                  (3, 13, 4, 5)]         # G = 4 at D = 4: R5
# (S, B, D, mode, reserve_sms): B above the grid and not a multiple of it
MOMENTS_SHAPES = [(2, 600, 8192, m, 0) for m in ("shared", "per_sample", "from_t2")] + [(2, 600, 8192, "from_t2", 20)] + \
                 [(2, 300, 16384, m, 0) for m in ("shared", "per_sample", "from_t2")] + \
                 [(2, 150, 32768, m, 0) for m in ("shared", "per_sample", "from_t2")] + [(2, 150, 32768, "per_sample", 7)]


def _stacked_dims(n_in, n_out):
    D = max(4, 1 << (n_in - 1).bit_length())
    return D, _cdiv(n_out, D)


def _loss_family(D, bias):
    return "loss_tm" if D >= 2048 and not bias else "loss"


# Cells every list must reach.  The forward runs several CTAs per SM (no waves in its plan), has no workspace slabs and
# no pass A / pass B: R3-R6 do not apply to it.  R6 is checked once, on the backward at D = 4 (the smallest workspace);
# pass A's grid-z loop does not depend on D or on which kernel filled the slabs.  Moments: every mode at every D, one
# call with reserve_sms > 0.
FAMILY_DIMS = {"fwd": [1 << k for k in FWD], "bwd": [1 << k for k in BWD], "loss": [1 << k for k in LOSS],
               "loss_tm": [1 << k for k in LOSS_TM]}
FAMILY_REGIMES = {"fwd": ("R1", "R2"), "bwd": ("R1", "R2", "R3", "R4", "R5"), "loss": ("R1", "R2", "R3", "R4", "R5"),
                  "loss_tm": ("R1", "R2", "R3", "R4", "R5")}
# cells that cannot occur: a tile of these kernels holds whole rows (D >= tile), so no tile is partial
UNREACHABLE = {("fwd", D, "R1"): "D >= tile" for D in (1024, 4096, 8192, 16384, 32768)}
UNREACHABLE.update({("bwd", D, "R1"): "D >= tile" for D in (1024, 4096, 8192)})
UNREACHABLE.update({("loss", D, "R1"): "D >= tile" for D in (1024, 2048, 4096)})
UNREACHABLE.update({("loss_tm", 4096, "R1"): "D >= tile"})


def covered_cells():
    cells = set()
    for S, B, D in FWD_SHAPES:
        cells |= {("fwd", D, r) for r in fwd_regimes(S, B, D)}
    for S, B, D in BWD_SHAPES + [R6_SHAPE]:
        cells |= {("bwd", D, r) for r in bwd_regimes(S, B, D)}
    for S, B, D, bias in LOSS_SHAPES:
        fam = _loss_family(D, bias)
        cells |= {(fam, D, r) for r in loss_regimes(S, B, D, fam == "loss_tm")}
    for n_in, n_out, S, B in STACKED_SHAPES:
        D, G = _stacked_dims(n_in, n_out)
        assert G > 1
        cells |= {("stacked", r) for r in bwd_regimes(S * G, B, D, groups=G)}
    for S, B, D, mode, reserve in MOMENTS_SHAPES:
        if moments_regimes(B, D, reserve):
            cells.add(("moments", D, mode))
            if reserve:
                cells.add(("moments", "reserve_sms"))
    return cells


def required_cells():
    cells = {(fam, D, r) for fam, dims in FAMILY_DIMS.items() for D in dims for r in FAMILY_REGIMES[fam]}
    cells -= set(UNREACHABLE)
    cells |= {("bwd", 4, "R6"), ("stacked", "R2"), ("stacked", "R4"), ("stacked", "R5"), ("moments", "reserve_sms")}
    cells |= {("moments", 1 << k, m) for k in MOMENTS_CTAS_PER_SM for m in ("shared", "per_sample", "from_t2")}
    return cells


def _size_grid():
    """(S, B, D) combinations for the size-query check: every shape of the lists plus a grid around the plans' break
    points (one tile, a multiple of min_iters tiles, just past one wave, S past the grid-z limit)."""
    shapes = {(S, B, D) for S, B, D in FWD_SHAPES + BWD_SHAPES + [R6_SHAPE]}
    shapes |= {(S, B, D) for S, B, D, _ in LOSS_SHAPES}
    shapes |= {(S, B, D) for S, B, D, _, _ in MOMENTS_SHAPES}
    for k in range(2, 16):
        for S in (1, 2, 3, 7, 37, 148, 149, 1024, 65539):
            for B in (1, 2, 5, 33, 65, 257, 1000, 4099):
                shapes.add((S, B, 1 << k))
    return sorted(shapes)


# ------------------------------------------------------------------------------------------------- CPU
def test_restated_plan_matches_library_queries():
    """The restatement above against the compiled library's size queries (no CUDA call is made).  A change of plan.cuh or of
    a launch table that is not carried over here fails this test, and with it the regime lists' coverage."""
    from ctypes import byref, c_int64, c_size_t
    from whvi_b200 import _lib
    L = _lib.lib()
    n = c_int64(0)
    ws, sq = c_size_t(0), c_int64(0)
    for S, B, D in _size_grid():
        k = _log2(D)
        _lib.check(L.whvi_layer_fwd_partials(S, B, D, byref(n)), "whvi_layer_fwd_partials")
        assert n.value == fwd_split(S, B, D).cps * S, (S, B, D)
        if k in BWD:
            _lib.check(L.whvi_layer_bwd_workspace_bytes(S, B, D, byref(ws)), "whvi_layer_bwd_workspace_bytes")
            assert ws.value == bwd_workspace_bytes(S, B, D), (S, B, D)
        if k in LOSS:
            _lib.check(L.whvi_layer_loss_sizes(S, B, D, byref(ws), byref(sq)), "whvi_layer_loss_sizes")
            assert (ws.value, sq.value) == loss_sizes(S, B, D), (S, B, D)
    stacked = [(S, B) + _stacked_dims(n_in, n_out) for n_in, n_out, S, B in STACKED_SHAPES]
    stacked += [(S, B, 1 << k, G) for k in BWD for S in (1, 3, 150) for B in (1, 7, 100) for G in (2, 5)]
    for S, B, D, G in stacked:
        for want_dx in (0, 1):
            _lib.check(L.whvi_stacked_bwd_workspace_bytes(S, B, D, G, want_dx, byref(ws)), "whvi_stacked_bwd_workspace_bytes")
            assert ws.value == stacked_bwd_workspace_bytes(S, B, D, G, want_dx), (S, B, D, G, want_dx)


def test_every_regime_cell_is_covered():
    covered, required = covered_cells(), required_cells()
    missing = sorted(required - covered, key=str)
    assert not missing, f"regime cells without a shape: {missing}"
    assert not set(UNREACHABLE) & covered
    for (fam, D, _), why in UNREACHABLE.items():   # the reason holds for the restated plan
        tile = 1 << {"fwd": FWD, "bwd": BWD, "loss": LOSS, "loss_tm": LOSS_TM}[fam][_log2(D)][0]
        assert why == "D >= tile" and D >= tile
    for S, B, D in FWD_SHAPES + BWD_SHAPES:
        assert S * B * D <= 1 << 24
    for S, B, D, _ in LOSS_SHAPES:
        assert S * B * D <= 1 << 24
    for S, B, D, _, _ in MOMENTS_SHAPES:
        assert S * B * D <= 1 << 24
    assert "R6" in bwd_regimes(*R6_SHAPE) and reduce_branches(R6_SHAPE[0], bwd_split(*R6_SHAPE), R6_SHAPE[2])[1] == 65535


# ------------------------------------------------------------------------------------------------- GPU helpers
def dev():
    return torch.device("cuda:0")


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev())


def _randn(rng, *shape):
    """fp32 draws widened to fp64: the oracle sees exactly the kernel's inputs."""
    return rng.standard_normal(shape, dtype=np.float32).astype(np.float64)


def _poison(*queries):
    """Fill the cached workspace with 0xFF bytes (NaN) before a call, at least as large as every size the call may ask
    for, so the call gets this very buffer: a slab that a kernel does not write reaches the sums as NaN."""
    from whvi_b200 import functional as F
    F._workspace(dev(), max(F._query(*q)[0] for q in queries)).fill_(255)


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=dev())


def _close(got, ref, what):
    err = rel_err(got.cpu().numpy() if isinstance(got, torch.Tensor) else got, ref)
    assert err < TOL, f"{what}: rel err {err}"


def _sum_close(got, ref, what):
    assert abs(float(got) - ref) < TOL * abs(ref), f"{what}: {float(got)} vs {ref}"


# ------------------------------------------------------------------------------------------------- fp32 vs the fp64 oracle
@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D", FWD_SHAPES)
def test_forward_vs_oracle(S, B, D):
    """layer_fwd into a NaN-filled output: per-sample x with bias, ReLU and the squared-error sum (added up from per-CTA
    partials); shared x without bias; the hoisted first transform (FROM_T2) with bias."""
    from oracle import oracle as O
    from whvi_b200 import functional as F
    from whvi_b200.fwht import fwht_
    rng = np.random.default_rng(S * 100003 + B * 31 + D)
    x, xs, g, s1, s2, bias, target = (_randn(rng, S, B, D), _randn(rng, B, D), _randn(rng, S, D), _randn(rng, D),
                                      _randn(rng, D), _randn(rng, D), _randn(rng, B, D))
    out = _nan(S, B, D)
    y, sq = F.layer_forward_raw(t(x), t(g), t(s1), t(s2), t(bias), out=out, relu_out=True, target=t(target))
    assert y is out
    ref = np.maximum(O.layer_fwd(x, g, s1, s2, bias), 0.0)
    _close(y, ref, "y (per-sample x, bias, relu)")
    _sum_close(sq, float(((ref - target[None]) ** 2).sum()), "sum (y - target)^2")
    ref = O.layer_fwd(xs, g, s1, s2)
    _close(F.layer_forward_raw(t(xs), t(g), t(s1), t(s2), out=_nan(S, B, D)), ref, "y (shared x)")
    t2 = fwht_(t(xs) * t(s2))
    y = F.layer_forward_raw(t2, t(g), t(s1), t(s2), t(bias), out=_nan(S, B, D), from_t2=True)
    _close(y, ref + bias, "y (from t2, bias)")


def _bwd_case(S, B, D):
    rng = np.random.default_rng(S * 7919 + B * 17 + D)
    return (_randn(rng, S, B, D), _randn(rng, B, D), _randn(rng, S, B, D), _randn(rng, S, D), _randn(rng, D), _randn(rng, D),
            _randn(rng, B, D))


def _check_bwd(got, ref, dx_mask, tag, dbias=True):
    dx, dg, ds1, ds2, db = got
    rdx, rdg, rds1, rds2, rdb = ref
    if dx_mask is not None:
        _close(dx, rdx * dx_mask, f"dx {tag}")
    for name, a, b in (("dg", dg, rdg), ("ds1", ds1, rds1), ("ds2", ds2, rds2)) + ((("dbias", db, rdb),) if dbias else ()):
        _close(a, b, f"{name} {tag}")


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D", BWD_SHAPES)
def test_backward_vs_oracle(S, B, D):
    """layer_bwd with the workspace poisoned: per-sample x with the ReLU mask on dx and a dy scale; then the RESID form
    (dy = coef * (saved output - target)) on a shared x without dx."""
    from oracle import oracle as O
    from whvi_b200 import functional as F
    x, xs, dy, g, s1, s2, target = _bwd_case(S, B, D)
    q = ("whvi_layer_bwd_workspace_bytes", S, B, D)
    _poison(q)
    got = F.layer_backward_raw(t(x), t(dy), t(g), t(s1), t(s2), want_dx=True, want_dbias=True, relu_in=True,
                               dy_scale=torch.tensor([0.375], device=dev()))
    _check_bwd(got, O.layer_bwd(x, 0.375 * dy, g, s1, s2, want_dbias=True), x > 0, "(per-sample x, relu_in, dy_scale)")
    _poison(q)
    got = F.layer_backward_raw(t(xs), t(dy), t(g), t(s1), t(s2), want_dx=False, want_dbias=True, target=t(target),
                               coef=torch.tensor(0.375, device=dev()))
    assert got[0] is None
    _check_bwd(got, O.layer_bwd(xs, 0.375 * (dy - target[None]), g, s1, s2, want_dbias=True), None, "(RESID, shared x)")


@pytest.mark.gpu
def test_backward_more_than_65535_samples():
    """R6: pass A covers samples past grid z = 65535 by looping (about 4.3 GB of workspace)."""
    from oracle import oracle as O
    from whvi_b200 import functional as F
    S, B, D = R6_SHAPE
    x, _, dy, g, s1, s2, _ = _bwd_case(S, B, D)
    try:
        _poison(("whvi_layer_bwd_workspace_bytes", S, B, D))
        got = F.layer_backward_raw(t(x), t(dy), t(g), t(s1), t(s2), want_dx=True, want_dbias=True)
        _check_bwd(got, O.layer_bwd(x, dy, g, s1, s2, want_dbias=True), 1.0, f"S={S}")
    finally:   # do not keep a 4.3 GB cached workspace around for the rest of the session
        F._WORKSPACES.clear()
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D,bias", LOSS_SHAPES)
def test_loss_layer_vs_oracle(S, B, D, bias):
    """layer_loss (forward + residual + backward for a unit coefficient) with the workspace poisoned."""
    from oracle import oracle as O
    from whvi_b200 import functional as F
    x, _, _, g, s1, s2, target = _bwd_case(S, B, D)
    bv = _randn(np.random.default_rng(D), D) if bias else None
    _poison(("whvi_layer_loss_sizes", S, B, D))
    sq, dx, dg, ds1, ds2, db = F.layer_loss_raw(t(x), t(g), t(s1), t(s2), None if bv is None else t(bv), t(target),
                                                want_dx=True, relu_in=True)
    r = O.layer_fwd(x, g, s1, s2, bv) - target[None]
    _sum_close(sq, float((r ** 2).sum()), "sum r^2")
    rdx, rdg, rds1, rds2, rdb = O.layer_bwd(x, r, g, s1, s2, want_dbias=True)
    assert (db is not None) == bias
    _check_bwd((dx, dg, ds1, ds2, db), (rdx, rdg, rds1, rds2, rdb), x > 0, f"bias={bias}", dbias=bias)


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D,mode,reserve", MOMENTS_SHAPES)
def test_layer_moments_vs_oracle(S, B, D, mode, reserve):
    """layer_moments with more rows than CTAs (each CTA resets its tensor-memory sums between rows): overwrite with a
    bias into NaN-filled sums, accumulate a second call, then the init= form (out = in + sums) into NaN-filled sums."""
    from oracle import oracle as O
    from whvi_b200 import functional as F
    from whvi_b200.fwht import fwht_
    rng = np.random.default_rng(D + 31 * B + len(mode) + reserve)
    x = _randn(rng, S, B, D) if mode == "per_sample" else _randn(rng, B, D)
    g, s1, s2, bias = _randn(rng, S, D), _randn(rng, D), _randn(rng, D), _randn(rng, D)
    g2 = g[::-1].copy()
    xin = fwht_(t(x) * t(s2)) if mode == "from_t2" else t(x)
    kw = dict(from_t2=mode == "from_t2", reserve_sms=reserve)
    y = O.layer_fwd(x, g, s1, s2, bias)
    y2 = O.layer_fwd(x, g2, s1, s2)
    sy, sy2 = _nan(B, D), _nan(B, D)
    F.layer_moments_raw(xin, t(g), t(s1), t(s2), t(bias), sy, sy2, **kw)
    _close(sy, y.sum(0), "sum y")
    _close(sy2, (y * y).sum(0), "sum y^2")
    F.layer_moments_raw(xin, t(g2), t(s1), t(s2), None, sy, sy2, accumulate=True, **kw)
    a, b = y.sum(0) + y2.sum(0), (y * y).sum(0) + (y2 * y2).sum(0)
    _close(sy, a, "sum y (accumulated)")
    _close(sy2, b, "sum y^2 (accumulated)")
    oy, oy2 = _nan(B, D), _nan(B, D)
    F.layer_moments_raw(xin, t(g), t(s1), t(s2), t(bias), oy, oy2, init=(sy, sy2), **kw)
    _close(oy, a + y.sum(0), "in + sum y")
    _close(oy2, b + (y * y).sum(0), "in + sum y^2")


@pytest.mark.gpu
@pytest.mark.parametrize("n_in,n_out,S,B", STACKED_SHAPES)
def test_grouped_stacked_vs_oracle(n_in, n_out, S, B):
    """One grouped Stacked call per direction (G blocks as virtual samples, parameters picked per group, the reduction's
    per-group sums) against the oracle block by block: pad x to D, run each block, concatenate and crop; pad dy per block,
    sum the blocks' dx."""
    from oracle import oracle as O
    from whvi_b200 import functional as F
    D, G = _stacked_dims(n_in, n_out)
    rng = np.random.default_rng(n_in * 13 + n_out)
    x, dy, g = _randn(rng, S, B, n_in), _randn(rng, S, B, n_out), _randn(rng, G, S, D)
    s1, s2, bias = _randn(rng, G, D), _randn(rng, G, D), _randn(rng, G * D)
    xt, gt, bt = t(x).requires_grad_(), t(g).requires_grad_(), t(bias).reshape(1, G * D).requires_grad_()
    s1t = [t(v).requires_grad_() for v in s1]
    s2t = [t(v).requires_grad_() for v in s2]
    y = F.whvi_stacked_g(xt, gt, bt, n_out, s1t, s2t)
    _poison(("whvi_stacked_bwd_workspace_bytes", S, B, D, G, 1))
    dx, dg, db, *ds = torch.autograd.grad(y, [xt, gt, bt] + s1t + s2t, t(dy))
    xp = np.zeros((S, B, D))
    xp[..., :n_in] = x
    dyp = np.zeros((S, B, G * D))
    dyp[..., :n_out] = dy
    blocks = [O.layer_bwd(xp, dyp[..., k * D:(k + 1) * D], g[k], s1[k], s2[k], want_dbias=True) for k in range(G)]
    yref = np.concatenate([O.layer_fwd(xp, g[k], s1[k], s2[k], bias[k * D:(k + 1) * D]) for k in range(G)], axis=-1)
    _close(y.detach(), yref[..., :n_out], "y")
    _close(dx, sum(b[0] for b in blocks)[..., :n_in], "dx")
    _close(dg, np.stack([b[1] for b in blocks]), "dg")
    _close(torch.stack(ds[:G]), np.stack([b[2] for b in blocks]), "ds1")
    _close(torch.stack(ds[G:]), np.stack([b[3] for b in blocks]), "ds2")
    _close(db.reshape(-1), np.concatenate([b[4] for b in blocks]), "dbias")


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D", [(2, 1793, 128), (2, 113, 4096), (2, 73, 8192)])
def test_reductions_are_bit_reproducible(S, B, D):
    """The fixed-order reductions give the same bits twice, with the workspace poisoned again in between: the backward and
    the loss layer at several CTAs per sample and >= 9 slabs per sample (R2, R4), and the forward's squared-error sum."""
    from whvi_b200 import functional as F
    assert {"R2", "R4"} <= bwd_regimes(S, B, D) and "R2" in fwd_regimes(S, B, D)
    x, _, dy, g, s1, s2, target = _bwd_case(S, B, D)
    runs = []
    for _ in range(2):
        _poison(("whvi_layer_bwd_workspace_bytes", S, B, D))
        out = list(F.layer_backward_raw(t(x), t(dy), t(g), t(s1), t(s2), want_dx=True, want_dbias=True))
        out.append(F.layer_forward_raw(t(x), t(g), t(s1), t(s2), target=t(target))[1])
        if D <= 4096:
            _poison(("whvi_layer_loss_sizes", S, B, D))
            out += [v for v in F.layer_loss_raw(t(x), t(g), t(s1), t(s2), t(s1), t(target)) if v is not None]
        runs.append(out)
    for i, (a, b) in enumerate(zip(*runs)):
        assert torch.equal(a, b), f"output {i} differs between two identical calls"


# ------------------------------------------------------------------------------------------------- bf16 twins
BF16_SHAPES = [s for s in BWD_SHAPES if bwd_regimes(*s) & {"R1", "R2", "R3", "R4"}]
BF16_LOSS_SHAPES = [s for s in LOSS_SHAPES if loss_regimes(*s[:3], _loss_family(s[2], s[3]) == "loss_tm") & {"R1", "R2", "R3", "R4"}]


def _eq(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    assert torch.equal(a, b), f"{what}: max |diff| {(a.float() - b.float()).abs().max().item()}"


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D", BF16_SHAPES)
def test_bf16_forward_backward_are_fp32_on_widened_inputs(S, B, D):
    """The bf16 forward and backward at the multi-CTA shapes equal the fp32 kernels (pinned to the oracle above) on the
    widened inputs: y and dx rounded once, the parameter gradients bit for bit.  D = 4 with an odd B takes the padded
    backward."""
    from whvi_b200 import functional as F
    x, _, dy, g, s1, s2, _ = _bwd_case(S, B, D)
    xb, dyb = t(x).to(torch.bfloat16), t(dy).to(torch.bfloat16)
    y16 = F.layer_forward_bf16(xb, t(g), t(s1), t(s2), t(s1), relu_out=True)
    _eq(y16, F.layer_forward_raw(xb.float(), t(g), t(s1), t(s2), t(s1), relu_out=True).to(torch.bfloat16), "y")
    sc = torch.tensor([0.375], device=dev())
    q = [("whvi_layer_bwd_workspace_bytes", S, B, D), ("whvi_layer_bwd_workspace_bytes", S, B + 1, D)]
    _poison(*q)
    b16 = F.layer_backward_raw(xb, dyb, t(g), t(s1), t(s2), want_dx=True, want_dbias=True, relu_in=True, dy_scale=sc)
    _poison(*q)
    b32 = F.layer_backward_raw(xb.float(), dyb.float(), t(g), t(s1), t(s2), want_dx=True, want_dbias=True, relu_in=True,
                               dy_scale=sc)
    _eq(b16[0], b32[0].to(torch.bfloat16), "dx")
    for name, a, b in zip(("dg", "ds1", "ds2", "dbias"), b16[1:], b32[1:]):
        _eq(a, b, name)


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,D,bias", BF16_LOSS_SHAPES)
def test_bf16_loss_layer_is_fp32_on_widened_inputs(S, B, D, bias):
    from whvi_b200 import functional as F
    x, _, _, g, s1, s2, target = _bwd_case(S, B, D)
    xb = t(x).to(torch.bfloat16)
    bv = t(s2) if bias else None
    outs = []
    for xin in (xb, xb.float()):
        _poison(("whvi_layer_loss_sizes", S, B, D))
        outs.append(F.layer_loss_raw(xin, t(g), t(s1), t(s2), bv, t(target), want_dx=True, relu_in=True))
    (sq16, dx16, *p16), (sq32, dx32, *p32) = outs
    _eq(sq16, sq32, "sum r^2")
    _eq(dx16, dx32.to(torch.bfloat16), "dx")
    for name, a, b in zip(("dg", "ds1", "ds2", "dbias"), p16, p32):
        if a is not None:
            _eq(a, b, name)
