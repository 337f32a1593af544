"""The FWHT and dense-posterior kernels against fp64 in every work-split regime they run in.

csrc/fwht.cu (kernel (1): the single-pass transform in fp32, bf16 and scaled form, the tiny kernel for D <= 2 and the multi-pass
schedule past 2^15), csrc/fwht_f64.cu (the fp64 transform) and csrc/reparam_dense.cu (the dense reparameterisation as a tcgen05
GEMM split into triangle units, its mode-1 dL GEMM, the small-D CUDA-core kernels and the dense KL, plain and grouped) cut
their work with host-side rules.  This file restates those rules from the source (CPU, with the cited lines checked), pins the
workspace sizes to the library's queries, checks that the restated unit map partitions the triangle, picks shapes that reach
each regime and checks that every (kernel, regime) cell has one.  A census ties every kernel under csrc/ to the test file that
checks its regimes.  On the GPU the kernels run at those shapes against fp64 with every output and workspace filled with NaN
first (in-place transforms excepted), so an element, tile, unit or sample block a kernel skips shows up as NaN or a large
error.

References.  FWHT: ``O.fwht`` (fp64), and for calls past 2^31 elements a torch fp64 FWHT built from reshapes (``fwht_t``),
run on the device chunk by chunk; a CPU test ties it to ``O.fwht``.  Dense forward: ``mu + eps @ tril(L)^T`` in torch fp64
(``dense_fwd_ref``), tied to ``O.reparam(dense=True)``.  Dense backward: ``tril(dg^T eps)`` and ``sum_s dg`` in torch fp64,
tied to ``O.reparam_dense_bwd``.  Dense KL: ``O.kl_dense``, and at D = 16384 its torch fp64 restatement ``kl_dense_ref``,
tied to ``O.kl_dense``; the grouped KL is the sum of the per-block KLs.

Tolerances are max|got - ref| / max|ref| (``rel_err``) unless a test says otherwise: 1e-5 for the transforms, the dense
forward and the KL; sums over S samples (dL, dmu) 1e-5 of max(max|ref|, sqrt(S)) (``sum_err``: a cancelled fp32 sum is only
as exact as its terms); fp64 transforms 1e-13.  The tcgen05 GEMM's outputs past a contraction of 1024 (the dense forward
at D >= 16384, dL at S > 1024) are bounded by the worst case of their accumulation chain instead (``gemm_tol``).
"""
from __future__ import annotations

import re
from pathlib import Path

import numpy as np
import pytest
import torch

from conftest import rel_err

SMS = 148
TESTS = Path(__file__).resolve().parent
CSRC = TESTS.parent / "whvi_b200" / "csrc"


def _cdiv(a, b):
    return -(-a // b)


def _round_up(v, m):
    return _cdiv(v, m) * m


# ------------------------------------------------------------------------------------------------- FWHT launch rules, restated
# fwht.cu: K = log2 D -> (N, C, GROUPS) of launch_cfg; a tile is 2^N elements, a CTA holds GROUPS tiles of 2^(N - C) threads.
# launch_fwht_single (D <= 2^15, fp32 and bf16) and launch_fwht_scaled (4 <= D <= 2^15) use the same table.
FWHT_CFG = {**{k: (10, 5, 8) for k in range(2, 11)}, 11: (11, 5, 4), 12: (12, 5, 2), 13: (13, 5, 1), 14: (14, 6, 1),
            15: (15, 6, 1)}
FWHT_SINGLE_LINES = {2: 216, 3: 217, 4: 218, 5: 219, 6: 220, 7: 221, 8: 222, 9: 223, 10: 224, 11: 226, 12: 227, 13: 228,
                     14: 230, 15: 231}
FWHT_SCALED_LINES = {k: 181 + k for k in range(2, 16)}
TINY_THREADS = 256            # fwht.cu:209: fwht_tiny_kernel, one row per thread, 256 rows per CTA, for K <= 1 (:208)
MAX_LOG2_SINGLE = 15


def fwht_launch(k, rows):
    """fwht.cu:170-172: tiles = ceil(total / 2^N), CTAs = ceil(tiles / GROUPS); at N = 15 with GROUPS = 1 the grid is
    persistent, capped at 148 CTAs that loop over tiles (:35, :38-40).  Returns (N, C, GROUPS, tiles, CTAs launched, threads)."""
    N, C, G = FWHT_CFG[k]
    total = rows << k
    tiles = _cdiv(total, 1 << N)
    ctas = _cdiv(tiles, G)
    if N >= 15 and G == 1:
        ctas = min(ctas, SMS)
    return N, C, G, tiles, ctas, (1 << (N - C)) * G


def fwht_persistent(k):
    N, _, G = FWHT_CFG[k]
    return N >= 15 and G == 1


def fwht_one_round(k):
    """fwht.cu:27: kOneRound = K <= 2 (the first butterfly round covers every bit, no transposition)."""
    return k <= 2


def tiny_ctas(rows):
    return _cdiv(rows, TINY_THREADS)


def multipass_schedule(k):
    """fwht.cu:255-259: for D > 2^15 the low 15 bits in one persistent pass over 2^15-element segments, then the high bits in
    passes of r = min(4, K - b) bits."""
    rs, b = [], MAX_LOG2_SINGLE
    while b < k:
        r = min(4, k - b)
        rs.append(r)
        b += r
    return rs


# fwht_f64.cu
SEG_LOG2 = 12


def f64_seg_k(k):
    """fwht_f64.cu:54: a segment is 2^seg_k doubles: 256 for k < 8 (several rows), the row for 8 <= k <= 12, 4096 above."""
    return (8 if k < 8 else k) if k < SEG_LOG2 else SEG_LOG2


def f64_stage_passes(k):
    """fwht_f64.cu:62: one global radix-2 stage per bit b in [12, k)."""
    return max(0, k - SEG_LOG2)


# ------------------------------------------------------------------------------------------------- dense launch rules, restated
BM, BK = 128, 32   # reparam_dense.cu:33-34: 128 rows (TMEM lanes) per unit, 32 fp32 per K block


def dense_q(D):
    """reparam_dense.cu:323-334: column blocks per unit, from 4 doubling until the triangle has at most 3 x 148 units or
    q >= RB."""
    RB = D // BM
    q = 4
    while True:
        if dense_units(D, q) <= SMS * 3 or q >= RB:
            return q
        q *= 2


def dense_units(D, q=None):
    """reparam_dense.cu:355-356: row block rb has rb // q + 1 units."""
    q = dense_q(D) if q is None else q
    return sum(rb // q + 1 for rb in range(D // BM))


def tri_unit(u, q):
    """reparam_dense.cu:85-92."""
    g = 0
    while q * (g + 1) * (g + 2) // 2 <= u:
        g += 1
    r = u - q * g * (g + 1) // 2
    return g * q + r // (g + 1), r % (g + 1)


def tri_unit_base(rb, q):
    """reparam_dense.cu:93-97."""
    g = rb // q
    return q * g * (g + 1) // 2 + (rb - g * q) * (g + 1)


def unit_k_blocks(rb, chunk, q):
    """reparam_dense.cu:117-119: a unit's K blocks [chunk q 4, min((chunk + 1) q, rb + 1) 4)."""
    return chunk * q * (BM // BK), min((chunk + 1) * q, rb + 1) * (BM // BK)


def sample_blocks(S):
    """reparam_dense.cu:359-361: samples in blocks of up to 256, each padded to NP = round_up(ns, 16) (the MMA's N)."""
    return [(s0, min(256, S - s0), _round_up(min(256, S - s0), 16)) for s0 in range(0, S, 256)]


def dense_stages(n):
    """reparam_dense.cu:315: a 3-stage mbarrier ring when n <= 128, else 2."""
    return 3 if n <= 128 else 2


def tm_cols(n):
    """reparam_dense.cu:110-111: TMEM columns, the next power of two >= n from 32."""
    c = 32
    while c < n:
        c <<= 1
    return c


def single_unit(rb, q):
    """reparam_dense.cu:228: a row block with rb < q is one unit and writes G itself; the others go through the reduce kernel
    (:365-366, grid (RB - q, ns))."""
    return rb < q


def mode1_grid(Sp, D):
    """reparam_dense.cu:382-383: the dL GEMM has RB (RB + 1) / 2 lower-triangle tiles, each a contraction of Sp / 32 K blocks."""
    RB = D // BM
    return RB * (RB + 1) // 2, Sp // BK


def small_st(D):
    """reparam_dense.cu:587: samples per CTA of reparam_dense_small_kernel (grid (ceil(S / ST), G), :588)."""
    return 4096 // D if D >= 16 else 256


def small_bwd_ctas(D):
    """reparam_dense.cu:602: reparam_dense_small_bwd_kernel has one thread per output of D * D + D, 256 per CTA; samples in
    tiles of 32 (:498, :519-520)."""
    return _cdiv(D * D + D, 256)


def kl_dense_threads(D):
    """reparam_dense.cu:449-452: the plain row kernel has 256 threads; the final kernel the next power of two >= D in
    [32, 1024], walking i += blockDim past that."""
    t = 32
    while t < D and t < 1024:
        t <<= 1
    return 256, t


def kl_dense_grouped_threads(D):
    """reparam_dense.cu:695-700: grouped row kernel 256 threads from D = 256, else 32; the final kernel as plain."""
    return (256 if D >= 256 else 32), kl_dense_threads(D)[1]


def dense_ws_bytes(S, D):
    """reparam_dense.cu:336-345: partial accumulators [unit][NP of the first sample block][128]."""
    NP = _round_up(min(S, 256), 16)
    return 4 * dense_units(D) * NP * BM


def dense_grouped_ws_bytes(S, D):
    """reparam_dense.cu:575-581: 0 below 128; else the larger of the forward's and the backward's two (D, round_up(S, 32))
    transposes."""
    if D < BM:
        return 0
    return max(dense_ws_bytes(S, D), 4 * 2 * D * _round_up(max(S, 1), BK))


# each restatement above, and the source text it rests on
CITED = ([("fwht.cu", ln, f"case {k}: return launch_cfg<{FWHT_CFG[k][0]}, {FWHT_CFG[k][1]}, {k}, {FWHT_CFG[k][2]}>(in, out, total, stream);")
          for k, ln in FWHT_SINGLE_LINES.items()] +
         [("fwht.cu", ln, f"case {k}: return launch_cfg<{FWHT_CFG[k][0]}, {FWHT_CFG[k][1]}, {k}, {FWHT_CFG[k][2]}, float, true>(")
          for k, ln in FWHT_SCALED_LINES.items()] +
         [("fwht.cu", 27, "constexpr bool kOneRound = (K <= 2);"),
          ("fwht.cu", 35, "constexpr bool PERSIST = (N >= 15) && GROUPS == 1;"),
          ("fwht.cu", 38, "const int64_t step = PERSIST ? int64_t(gridDim.x) * GROUPS * TILE : total;"),
          ("fwht.cu", 40, "base < total; base += step"),
          ("fwht.cu", 170, "const int64_t tiles = (total + (int64_t(1) << N) - 1) >> N;"),
          ("fwht.cu", 171, "int64_t ctas = (tiles + GROUPS - 1) / GROUPS;"),
          ("fwht.cu", 172, "if (N >= 15 && GROUPS == 1 && ctas > 148) ctas = 148;"),
          ("fwht.cu", 208, "if (K <= 1) {"),
          ("fwht.cu", 209, "const int threads = 256;"),
          ("fwht.cu", 210, "const int64_t blocks = (rows + threads - 1) / threads;"),
          ("fwht.cu", 255, "launch_cfg<15, 6, 15, 1>(in, out, total, stream)"),
          ("fwht.cu", 257, "const int r = (K - b) < 4 ? (K - b) : 4;"),
          ("fwht_f64.cu", 10, "constexpr int kSegLog2 = 12;"),
          ("fwht_f64.cu", 54, "int seg_k = k < kSegLog2 ? (k < 8 ? 8 : k) : kSegLog2;"),
          ("fwht_f64.cu", 62, "for (int b = kSegLog2; b < k; ++b) {"),
          ("reparam_dense.cu", 33, "constexpr int DG_BM = 128;"),
          ("reparam_dense.cu", 34, "constexpr int DG_BK = 32;"),
          ("reparam_dense.cu", 88, "while (q * (g + 1) * (g + 2) / 2 <= u) ++g;"),
          ("reparam_dense.cu", 89, "const int r = u - q * g * (g + 1) / 2;"),
          ("reparam_dense.cu", 90, "rb = g * q + r / (g + 1);"),
          ("reparam_dense.cu", 91, "chunk = r % (g + 1);"),
          ("reparam_dense.cu", 96, "return q * g * (g + 1) / 2 + (rb - g * q) * (g + 1);"),
          ("reparam_dense.cu", 110, "uint32_t tm_cols = 32;"),
          ("reparam_dense.cu", 111, "while (tm_cols < uint32_t(N)) tm_cols <<= 1;"),
          ("reparam_dense.cu", 117, "kb0 = chunk * p.q * (DG_BM / DG_BK);"),
          ("reparam_dense.cu", 118, "const int kend = min((chunk + 1) * p.q, row_blk + 1) * (DG_BM / DG_BK);"),
          ("reparam_dense.cu", 228, "const bool single = row_blk < p.q;"),
          ("reparam_dense.cu", 273, "const int base = tri_unit_base(rb, q), cnt = rb / q + 1;"),
          ("reparam_dense.cu", 315, "const int stages = a.n <= 128 ? 3 : 2;"),
          ("reparam_dense.cu", 326, "int q = 4;"),
          ("reparam_dense.cu", 329, "for (int64_t rb = 0; rb < RB; ++rb) units += rb / q + 1;"),
          ("reparam_dense.cu", 330, "if (units <= 148 * 3 || q >= RB) break;"),
          ("reparam_dense.cu", 331, "q *= 2;"),
          ("reparam_dense.cu", 342, "const int64_t ns = S < 256 ? S : 256;"),
          ("reparam_dense.cu", 343, "const int64_t NP = (ns + 15) / 16 * 16;"),
          ("reparam_dense.cu", 344, "return sizeof(float) * size_t(units) * NP * DG_BM;"),
          ("reparam_dense.cu", 359, "for (int64_t s0 = 0; s0 < S; s0 += 256)"),
          ("reparam_dense.cu", 361, "const int NP = (ns + 15) / 16 * 16;"),
          ("reparam_dense.cu", 365, "if (RB > q) {"),
          ("reparam_dense.cu", 366, "dim3 grid(static_cast<unsigned>(RB - q), static_cast<unsigned>(ns));"),
          ("reparam_dense.cu", 382, "static_cast<int>(Sp / DG_BK)"),
          ("reparam_dense.cu", 383, "RB * (RB + 1) / 2"),
          ("reparam_dense.cu", 449, "kl_dense_rows_kernel<<<static_cast<unsigned>(D), 256, 0, stream>>>"),
          ("reparam_dense.cu", 452, "while (threads < D && threads < 1024) threads <<= 1;"),
          ("reparam_dense.cu", 498, "constexpr int RDS_TILE_S = 32;"),
          ("reparam_dense.cu", 579, "const size_t bwd = sizeof(float) * 2 * size_t(D) * size_t(round_up(S < 1 ? 1 : S, DG_BK));"),
          ("reparam_dense.cu", 587, "const int ST = static_cast<int>(D >= 16 ? 4096 / D : 256);"),
          ("reparam_dense.cu", 588, "(S + ST - 1) / ST"),
          ("reparam_dense.cu", 602, "(D * D + D + RDS_THREADS - 1) / RDS_THREADS"),
          ("reparam_dense.cu", 609, "const int64_t Sp = round_up(S, DG_BK);"),
          ("reparam_dense.cu", 695, "const int threads = D >= 256 ? 256 : 32;"),
          ("reparam_dense.cu", 700, "while (ft < D && ft < 1024) ft <<= 1;")])


# ------------------------------------------------------------------------------------------------- the shapes
# FWHT single pass: (variant, k, rows, in place).  variant "f32" whvi_fwht_f32, "bf16" whvi_fwht_bf16, "scaled"
# whvi_fwht_scaled_f32 (out of place only: its contract does not allow in == out, and its callers write a separate t2).
FWHT_SHAPES = []
for _v in ("f32", "bf16", "scaled"):
    FWHT_SHAPES += [(_v, 4, 197, False),         # partial tile: 64 rows per 1024-element tile
                    (_v, 10, 19, False),         # N = 10: 19 tiles over 3 CTAs of 8 groups, the last with 5 idle groups
                    (_v, 11, 9, False),          # N = 11: 9 tiles, CTAs of 4 groups
                    (_v, 12, 5, False),          # N = 12: 5 tiles, CTAs of 2 groups
                    (_v, 2, 1001, False),        # one round (D = 4), partial tile
                    (_v, 6, 200003, False)]      # 1563 CTAs of 256 threads: more than one wave
    FWHT_SHAPES += [(_v, 15, rows, ip) for rows in (100, 148, 1041) for ip in ((False, True) if _v != "scaled" else (False,))]
    if _v != "scaled":
        FWHT_SHAPES += [(_v, 0, 1000, False), (_v, 1, 1000, True)]   # tiny kernel, 4 CTAs
# calls of more than 2^31 elements: (variant, k, rows)
FWHT_LARGE = [("f32", 15, 65537), ("scaled", 15, 65537), ("bf16", 2, (1 << 29) + 1), ("bf16", 15, 65537)]
# multi-pass fp32 (D > 2^15): (k, rows, in place); every first pass has more than 148 segments of 2^15
MULTIPASS_SHAPES = [(16, 77, False), (17, 39, False), (18, 19, False), (19, 10, True), (20, 5, False), (21, 3, False),
                    (22, 2, True), (23, 1, False)]
# fp64: (k, rows)
F64_SHAPES = [(3, 100), (7, 5), (8, 3), (12, 3), (14, 3), (17, 2)]
# dense forward: (S, D, G, mu_stride, L_stride); G = 0 is whvi_reparam_dense_f32, G >= 1 whvi_reparam_dense_grouped_f32
DENSE_FWD_SHAPES = [(5, 128, 0, 0, 0),            # q = 4, every row block one unit, NP = 16
                    (37, 512, 0, 0, 0),           # q = 4, one unit per row block, NP = 48
                    (128, 640, 0, 0, 0),          # RB = 5: one reduced row block, NP = 128 (3 stages)
                    (131, 1024, 0, 0, 0),         # NP = 144 (2 stages)
                    (256, 4096, 0, 0, 0),         # NP = 256, 144 units
                    (600, 1024, 0, 0, 0),         # sample blocks 256, 256, 88
                    (16, 8192, 0, 0, 0),          # q = 8
                    (20, 16384, 0, 0, 0),         # q = 32: a unit streams 128 K blocks
                    (16, 32768, 0, 0, 0),         # q = 128: a unit streams 512 K blocks
                    (37, 256, 3, 260, 256 * 256 + 64),
                    (300, 640, 2, 644, 640 * 640 + 128)]
# dense backward: (S, D, G); G = 0 is whvi_reparam_dense_bwd_f32 on caller-padded transposes, else the grouped entry point
DENSE_BWD_SHAPES = [(20, 128, 1),                 # Sp / 32 = 1 K block, S % 32 != 0
                    (4096, 256, 2),               # 128 K blocks through the 3-stage ring
                    (50, 640, 3),
                    (40, 16384, 1),               # 8256 tiles
                    (100, 384, 0), (33, 1024, 0)]
# small-D grouped (D <= 64): (S, D, G, mu_stride, L_stride)
SMALL_SHAPES = [(1000, 16, 1, 16, 256),           # ST = 256: 4 CTAs, the last with 232 samples; 1000 % 32 = 8
                (1000, 64, 2, 64, 4096),          # ST = 64: 16 CTAs, the last with 40; backward's last CTA 64 of 256
                (300, 8, 3, 12, 72),              # ST = 256 (D < 16), strided G > 1
                (77, 48, 3, 52, 48 * 48 + 16)]    # D not a power of two, strided
# dense KL: (D, G, mu_stride, L_stride, grad_scale); G = 0 is whvi_kl_dense_f32
KL_DENSE_SHAPES = [(300, 0, 0, 0, 0.375),
                   (16384, 0, 0, 0, 1.0),
                   (100, 3, 104, 100 * 100 + 12, 2.5),     # grouped, 32-thread rows
                   (300, 2, 300, 300 * 300, 1.0),          # grouped, 256-thread rows
                   (2048, 2, 2052, 2048 * 2048 + 4, 0.375)]  # grouped, final kernel walks 2 strides
# whvi_mc_moments_strided_f32: (S, n, y_sample_stride, accumulate)
MC_MOMENTS_SHAPES = [(3, 1028, 1028, False), (9, 4100, 4104, True), (4, 65540, 65540, True)]


# ------------------------------------------------------------------------------------------------- regimes
def fwht_cells(variant, k, rows, inplace):
    c = set()
    if k <= 1:
        if tiny_ctas(rows) > 1:
            c.add((variant, "tiny kernel, several CTAs"))
        return c
    N, C, G, tiles, ctas, threads = fwht_launch(k, rows)
    if (rows << k) % (1 << N):
        c.add((variant, "partial tile"))
    if G > 1 and tiles % G:
        c.add((variant, f"partial last CTA with idle groups, N = {N}"))
    if not fwht_persistent(k) and ctas > SMS * (2048 // threads):
        c.add((variant, "more than one wave"))
    if fwht_one_round(k):
        c.add((variant, "one round"))
    if fwht_persistent(k):
        where = "in place" if inplace else "out of place"
        if tiles < SMS:
            c.add((variant, f"persistent, tiles < 148, {where}"))
        elif tiles == SMS:
            c.add((variant, f"persistent, tiles = 148, {where}"))
        elif tiles % SMS:
            c.add((variant, f"persistent, tiles >> 148, tiles % 148 != 0, {where}"))
    if rows << k > 1 << 31:
        c.add((variant, "more than 2^31 elements"))
    return c


def multipass_cells(k, rows):
    c = set()
    if (rows << k) >> MAX_LOG2_SINGLE > SMS:
        c.add(("multipass", "first pass > 148 segments"))
    rs = multipass_schedule(k)
    c.add(("multipass", f"r = {rs[-1]}, only pass" if len(rs) == 1 else f"r = {rs[-1]}, tail"))
    return c


def f64_cells(k, rows):
    seg = f64_seg_k(k)
    if k < 8:
        per = 1 << (seg - k)
        return {("f64", "k < 8, rows % rows per segment != 0")} if rows % per else {("f64", "k < 8")}
    if k <= SEG_LOG2:
        return {("f64", "8 <= k <= 12")}
    return {("f64", "k > 12, stage passes")} if f64_stage_passes(k) else set()


def dense_fwd_cells(S, D, G, mu_stride, L_stride):
    q, RB = dense_q(D), D // BM
    c = {("dense_fwd", f"q = {q}" + (", every row block one unit" if RB <= q else ", reduce"))}
    if RB > q:
        c.add(("dense_fwd", "single-unit and reduced row blocks"))
    if RB == q + 1:
        c.add(("dense_fwd", "one reduced row block"))
    blocks = sample_blocks(S)
    for _, ns, NP in blocks:
        if NP == 16:
            c.add(("dense_fwd", "NP = 16"))
        elif NP < 128:
            c.add(("dense_fwd", "16 < NP < 128"))
        elif NP == 128 and dense_stages(NP) == 3:
            c.add(("dense_fwd", "NP = 128, 3 stages"))
        elif NP == 144 and dense_stages(NP) == 2:
            c.add(("dense_fwd", "NP = 144, 2 stages"))
        elif NP == 256:
            c.add(("dense_fwd", "NP = 256"))
    if len(blocks) > 1 and S % 256:
        c.add(("dense_fwd", "several sample blocks, ragged tail"))
    if G > 1 and mu_stride > D and L_stride > D * D:
        c.add(("dense_fwd", "grouped, mu_stride > D, L_stride > D D"))
    return c


def dense_bwd_cells(S, D, G):
    Sp = _round_up(S, BK)
    _, kb = mode1_grid(Sp, D)
    c = {("dense_bwd", "caller-padded transposes" if G == 0 else "grouped")}
    if kb == 1:
        c.add(("dense_bwd", "1 K block"))
    if kb >= 32 * dense_stages(BM):
        c.add(("dense_bwd", "K blocks >> stages"))
    if S % BK:
        c.add(("dense_bwd", "S % 32 != 0"))
    if D == 640:
        c.add(("dense_bwd", "D = 640"))
    if D >= 16384:
        c.add(("dense_bwd", "D >= 16384"))
    if G > 1:
        c.add(("dense_bwd", "G > 1"))
    return c


def small_cells(S, D, G, mu_stride, L_stride):
    c = set()
    st = small_st(D)
    if S > 2 * st and S % st:
        c.add(("small_d", "S >> ST, ragged last CTA"))
    if S % 32:
        c.add(("small_d", "ragged last 32-sample tile (backward)"))
    if D == 64 and (D * D + D) % 256:
        c.add(("small_d", "last backward CTA partly idle (D = 64)"))
    if G > 1 and mu_stride > D and L_stride > D * D:
        c.add(("small_d", "strided G > 1"))
    if D < 16:
        c.add(("small_d", "D < 16 (ST = 256)"))
    return c


def kl_dense_cells(D, G, mu_stride, L_stride, grad_scale):
    c = set()
    if G == 0:
        c.add(("kl_dense", "plain"))
        if D >= 16384:
            c.add(("kl_dense", "plain, D = 16384"))
    else:
        rows, final = kl_dense_grouped_threads(D)
        c.add(("kl_dense", f"grouped, {rows}-thread rows"))
        if final < D and G > 1:
            c.add(("kl_dense", "final kernel strided walk, G > 1"))
        if G > 1 and mu_stride > D and L_stride > D * D:
            c.add(("kl_dense", "grouped, strided"))
    if grad_scale != 1.0:
        c.add(("kl_dense", "grad_scale != 1"))
    return c


def mc_moments_cells(S, n, stride, accumulate):
    c = {("mc_moments", "4-sample loop and tail" if S > 4 and S % 4 else "tail only" if S < 4 else "4-sample loop only")}
    if (n // 4) % 256:
        c.add(("mc_moments", "last CTA partly idle"))
    if stride > n:
        c.add(("mc_moments", "sample stride > n"))
    c.add(("mc_moments", "accumulate" if accumulate else "no input sums"))
    return c


def covered_cells():
    cells = set()
    for v, k, rows, ip in FWHT_SHAPES:
        cells |= fwht_cells(v, k, rows, ip)
    for v, k, rows in FWHT_LARGE:
        cells |= fwht_cells(v, k, rows, False)
    for k, rows, _ in MULTIPASS_SHAPES:
        cells |= multipass_cells(k, rows)
    for k, rows in F64_SHAPES:
        cells |= f64_cells(k, rows)
    for shape in DENSE_FWD_SHAPES:
        cells |= dense_fwd_cells(*shape)
    for shape in DENSE_BWD_SHAPES:
        cells |= dense_bwd_cells(*shape)
    for shape in SMALL_SHAPES:
        cells |= small_cells(*shape)
    for shape in KL_DENSE_SHAPES:
        cells |= kl_dense_cells(*shape)
    for shape in MC_MOMENTS_SHAPES:
        cells |= mc_moments_cells(*shape)
    return cells


_FWHT_REQUIRED = ["partial tile", "partial last CTA with idle groups, N = 10", "partial last CTA with idle groups, N = 11",
                  "partial last CTA with idle groups, N = 12", "more than one wave", "one round",
                  "tiny kernel, several CTAs", "more than 2^31 elements"] + \
                 [f"persistent, {t}, {w}" for t in ("tiles < 148", "tiles = 148", "tiles >> 148, tiles % 148 != 0")
                  for w in ("in place", "out of place")]
REQUIRED = ({(v, r) for v in ("f32", "bf16", "scaled") for r in _FWHT_REQUIRED} |
            {("multipass", "first pass > 148 segments")} |
            {("multipass", f"r = {r}, {w}") for r in (1, 2, 3, 4) for w in ("only pass", "tail")} |
            {("f64", "k < 8, rows % rows per segment != 0"), ("f64", "8 <= k <= 12"), ("f64", "k > 12, stage passes")} |
            {("dense_fwd", c) for c in ("q = 4, every row block one unit", "q = 4, reduce", "q = 8, reduce", "q = 32, reduce",
                                        "q = 128, reduce", "single-unit and reduced row blocks", "one reduced row block",
                                        "NP = 16", "16 < NP < 128", "NP = 128, 3 stages", "NP = 144, 2 stages", "NP = 256",
                                        "several sample blocks, ragged tail", "grouped, mu_stride > D, L_stride > D D")} |
            {("dense_bwd", c) for c in ("grouped", "caller-padded transposes", "1 K block", "K blocks >> stages",
                                        "S % 32 != 0", "D = 640", "D >= 16384", "G > 1")} |
            {("small_d", c) for c in ("S >> ST, ragged last CTA", "ragged last 32-sample tile (backward)",
                                      "last backward CTA partly idle (D = 64)", "strided G > 1", "D < 16 (ST = 256)")} |
            {("kl_dense", c) for c in ("plain", "plain, D = 16384", "grouped, 32-thread rows", "grouped, 256-thread rows",
                                       "final kernel strided walk, G > 1", "grouped, strided", "grad_scale != 1")} |
            {("mc_moments", c) for c in ("tail only", "4-sample loop and tail", "4-sample loop only", "last CTA partly idle",
                                         "sample stride > n", "accumulate", "no input sums")})
# cells that cannot occur, and why
UNREACHABLE = {("scaled", "tiny kernel, several CTAs"): "whvi_fwht_scaled_f32 takes D >= 4 only",
               **{("scaled", f"persistent, {t}, in place"): "whvi_fwht_scaled_f32 does not allow in == out"
                  for t in ("tiles < 148", "tiles = 148", "tiles >> 148, tiles % 148 != 0")}}

# every __global__ function under csrc/ -> the test file that checks it in every work-split regime it runs in
KERNEL_TESTS = {
    **{k: "test_work_split.py" for k in (
        "layer_fwd_kernel", "layer_bwd_tma_kernel", "layer_bwd_tm_kernel", "layer_bwd_reduce_slabs_kernel",
        "layer_bwd_reduce_fold_kernel", "layer_loss_kernel", "layer_loss_tm_kernel", "layer_moments_kernel",
        "stack_concat_kernel", "stack_split_kernel", "stack_sum_kernel")},
    **{k: "test_column_param_regimes.py" for k in (
        "column_dot_kernel", "column_outer_kernel", "column_dot_dx_kernel", "column_dw_kernel", "column_outer_dx_kernel",
        "column_dbias_kernel", "column_param_kernel", "column_ds1_kernel", "reparam_diag_kernel", "reparam_diag_bwd_kernel",
        "kl_kernel", "adam_kernel")},
    **{k: "test_classification.py" for k in (
        "categorical_nll_kernel", "categorical_total_kernel", "categorical_nll_bwd_kernel", "categorical_predictive_kernel")},
    **{k: "test_conv.py" for k in ("im2col_kernel", "col2im_kernel")},
    **{k: "test_fwht_dense_regimes.py" for k in (
        "fwht_kernel", "fwht_tiny_kernel", "fwht_strided_kernel", "fwht_f64_segment_kernel", "fwht_f64_stage_kernel",
        "dense_gemm_kernel", "dense_reparam_reduce_kernel", "kl_dense_rows_kernel", "kl_dense_final_kernel",
        "reparam_dense_small_kernel", "reparam_dense_small_bwd_kernel", "dense_transpose_pad_kernel", "dense_colsum_kernel",
        "kl_dense_grouped_rows_kernel", "kl_dense_grouped_final_kernel", "mc_moments_kernel")},
}


def kernel_census():
    """Names of the __global__ functions defined in csrc/*.cu and csrc/*.cuh (comments stripped; an optional
    __launch_bounds__(...) with nested parentheses skipped)."""
    names = set()
    for path in sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")):
        src = re.sub(r"//[^\n]*|/\*.*?\*/", "", path.read_text(), flags=re.S)
        for m in re.finditer(r"__global__\s+void\s+", src):
            i = m.end()
            if src.startswith("__launch_bounds__", i):
                i = src.index("(", i)
                depth = 0
                while True:
                    depth += {"(": 1, ")": -1}.get(src[i], 0)
                    i += 1
                    if depth == 0:
                        break
            names.add(re.match(r"\s*(\w+)\s*\(", src[i:]).group(1))
    return names


# ------------------------------------------------------------------------------------------------- CPU
def test_cited_launch_rules_are_the_source():
    """Each restated rule cites a line of csrc/; the line still says it."""
    for name, line, text in CITED:
        src = (CSRC / name).read_text().splitlines()
        assert text in src[line - 1], f"{name}:{line} no longer reads {text!r}: {src[line - 1]!r}"


def test_restated_dense_q_is_the_table():
    """dense_q as the design states it: 4 up to D = 4096 (every row block one unit up to 512), then 8, 32, 128."""
    want = {128: 4, 256: 4, 384: 4, 512: 4, 640: 4, 1024: 4, 2048: 4, 4096: 4, 8192: 8, 16384: 32, 32768: 128}
    assert {D: dense_q(D) for D in want} == want
    assert [D for D in want if D // BM <= dense_q(D)] == [128, 256, 384, 512]
    assert tm_cols(16) == 32 and tm_cols(48) == 64 and tm_cols(144) == 256 and tm_cols(256) == 256


def test_restated_workspace_matches_library_query():
    """The dense workspace sizes against whvi_reparam_dense_workspace_bytes and
    whvi_reparam_dense_grouped_workspace_bytes at every regime shape and on a grid of (S, D)."""
    from ctypes import byref, c_size_t
    from whvi_b200 import _lib
    L = _lib.lib()
    ws = c_size_t(0)
    shapes = {(S, D) for S, D, *_ in DENSE_FWD_SHAPES} | {(S, D) for S, D, _ in DENSE_BWD_SHAPES}
    shapes |= {(S, D) for S in (0, 1, 16, 17, 128, 129, 256, 257, 600, 4096) for D in (128, 640, 4096, 8192, 16384, 32768)}
    for S, D in sorted(shapes):
        _lib.check(L.whvi_reparam_dense_workspace_bytes(S, D, byref(ws)), "whvi_reparam_dense_workspace_bytes")
        assert ws.value == dense_ws_bytes(S, D), (S, D)
        _lib.check(L.whvi_reparam_dense_grouped_workspace_bytes(S, D, byref(ws)), "whvi_reparam_dense_grouped_workspace_bytes")
        assert ws.value == dense_grouped_ws_bytes(S, D), (S, D)
    for S, D, *_ in SMALL_SHAPES:
        _lib.check(L.whvi_reparam_dense_grouped_workspace_bytes(S, D, byref(ws)), "whvi_reparam_dense_grouped_workspace_bytes")
        assert ws.value == 0


def test_restated_tri_unit_partitions_the_triangle():
    """For every D = 128 RB up to 32768: units 0 .. units - 1 map one-to-one onto the (row block, chunk) pairs with rb / q + 1
    chunks per row block, in chunk order from tri_unit_base(rb); a row block's chunks cover its column blocks 0 .. rb once;
    the single-unit row blocks are exactly those with rb < q; the triangle has at most 3 x 148 units unless q >= RB."""
    for RB in range(1, 257):
        D = RB * BM
        q = dense_q(D)
        units = dense_units(D)
        assert units <= SMS * 3 or q >= RB, D
        pairs = [tri_unit(u, q) for u in range(units)]
        assert sorted(pairs) == [(rb, c) for rb in range(RB) for c in range(rb // q + 1)], D
        for u, (rb, c) in enumerate(pairs):
            assert tri_unit_base(rb, q) + c == u, (D, u)
        for rb in range(RB):
            cnt = rb // q + 1
            assert single_unit(rb, q) == (cnt == 1)
            covered = []
            for c in range(cnt):
                k0, k1 = unit_k_blocks(rb, c, q)
                assert k1 > k0, (D, rb, c)
                covered += range(k0, k1)
            assert covered == list(range((rb + 1) * (BM // BK))), (D, rb)


def test_every_regime_cell_is_covered():
    cells = covered_cells()
    missing = sorted(REQUIRED - cells - set(UNREACHABLE))
    assert not missing, f"regime cells without a shape: {missing}"
    assert not (set(UNREACHABLE) & cells), "a cell listed as unreachable has a shape"
    for k, rows, _ in MULTIPASS_SHAPES:
        assert k > MAX_LOG2_SINGLE
    for S, D, G, mu_stride, L_stride in DENSE_FWD_SHAPES + SMALL_SHAPES:   # legal grouped calls
        assert G <= 1 or (mu_stride >= D and L_stride >= D * D)
        assert D < BM or G <= 1 or (mu_stride % 4 == 0 and L_stride % 4 == 0)


def test_kernel_census():
    """Every __global__ function under csrc/ is in KERNEL_TESTS, and every file named there exists."""
    found = kernel_census()
    assert found == set(KERNEL_TESTS), (f"not in KERNEL_TESTS: {sorted(found - set(KERNEL_TESTS))}; "
                                        f"no longer in csrc/: {sorted(set(KERNEL_TESTS) - found)}")
    for f in set(KERNEL_TESTS.values()):
        assert (TESTS / f).is_file(), f


# ------------------------------------------------------------------------------------------------- fp64 restatements
def fwht_t(x):
    """Sylvester-order FWHT of the rows of an fp64 torch tensor, one reshape per bit (any device)."""
    rows, D = x.shape
    h = 1
    while h < D:
        y = x.reshape(rows, D // (2 * h), 2, h)
        x = torch.stack((y[:, :, 0] + y[:, :, 1], y[:, :, 0] - y[:, :, 1]), dim=2).reshape(rows, D)
        h *= 2
    return x


def _upper(r0, r1, D, device):
    return torch.arange(D, device=device)[None, :] > torch.arange(r0, r1, device=device)[:, None]


def _chunks(D, rows_per=2048):
    return [(r0, min(D, r0 + rows_per)) for r0 in range(0, D, rows_per)]


def dense_fwd_ref(mu, L, eps):
    """mu + eps @ tril(L)^T in fp64; whatever lies above the diagonal of L (NaN, inf) is never used."""
    D = L.shape[0]
    e = eps.double()
    g = torch.empty((eps.shape[0], D), dtype=torch.float64, device=eps.device)
    for r0, r1 in _chunks(D):
        Lc = torch.where(_upper(r0, r1, D, L.device), 0.0, L[r0:r1].double())
        g[:, r0:r1] = e @ Lc.T + mu[r0:r1].double()
    return g


def dense_bwd_ref_rows(eps, dg, r0, r1):
    """Rows r0:r1 of dL = tril(dg^T eps) in fp64."""
    Lc = dg[:, r0:r1].double().T @ eps.double()
    return torch.where(_upper(r0, r1, eps.shape[1], eps.device), 0.0, Lc)


def kl_dense_ref(mu, L, lam):
    """0.5 (D ln lambda - 2 sum ln L_ii - D + |tril L|_F^2 / lambda + |mu|^2 / lambda) in fp64."""
    D = L.shape[0]
    sq = 0.0
    for r0, r1 in _chunks(D):
        Lc = torch.where(_upper(r0, r1, D, L.device), 0.0, L[r0:r1].double())
        sq += float((Lc * Lc).sum())
    logd = float(torch.log(torch.diagonal(L).double()).sum())
    m2 = float((mu.double() ** 2).sum())
    return 0.5 * (D * np.log(lam) - 2.0 * logd - D + sq / lam + m2 / lam)


def kl_dense_grad_ref_rows(L, lam, r0, r1):
    """Rows r0:r1 of dL = tril(L) / lambda - diag(1 / L_ii), 0 above the diagonal."""
    D = L.shape[0]
    Lc = torch.where(_upper(r0, r1, D, L.device), 0.0, L[r0:r1].double()) / lam
    idx = torch.arange(r0, r1, device=L.device)
    Lc[idx - r0, idx] -= 1.0 / L[idx, idx].double()
    return Lc


def sum_err(got, ref, S):
    """max |got - ref| against the size of a sum of S unit-scale terms (sqrt(S)), or of the result where that is larger."""
    return float((got.double() - ref).abs().max() / max(float(ref.abs().max()), np.sqrt(S)))


def _worst(a, b):
    """The larger of two errors, NaN if either is NaN (Python's max(0.0, nan) is 0.0: a NaN chunk would drop out)."""
    return a if (a != a or a >= b) else b


def _poison_upper(L):
    """NaN, +inf and -inf above the diagonal of L (D, D), in turn along each row."""
    D = L.shape[0]
    for r0, r1 in _chunks(D):
        up = _upper(r0, r1, D, L.device)
        col = torch.arange(D, device=L.device)[None, :] % 3
        Lc = L[r0:r1]
        Lc.masked_fill_(up & (col == 0), float("nan"))
        Lc.masked_fill_(up & (col == 1), float("inf"))
        Lc.masked_fill_(up & (col == 2), float("-inf"))


def test_fwht_restatement_is_the_oracle():
    from oracle import oracle as O
    rng = np.random.default_rng(3)
    for k in (0, 1, 2, 5, 10):
        x = rng.standard_normal((7, 1 << k))
        assert rel_err(fwht_t(torch.from_numpy(x)).numpy(), O.fwht(x)) < 1e-14


def test_dense_restatements_are_the_oracle():
    """dense_fwd_ref, dense_bwd_ref_rows, kl_dense_ref and kl_dense_grad_ref_rows against O.reparam(dense=True),
    O.reparam_dense_bwd and O.kl_dense (torch on the CPU, with NaN and inf above the diagonal of L and rows chunked)."""
    from oracle import oracle as O
    rng = np.random.default_rng(5)
    S, D, lam = 9, 2304, 0.3
    mu, eps, dg = rng.standard_normal(D), rng.standard_normal((S, D)), rng.standard_normal((S, D))
    L = np.tril(rng.standard_normal((D, D))) / np.sqrt(D)
    L[np.arange(D), np.arange(D)] = np.abs(np.diagonal(L)) + 0.1
    Lt = torch.from_numpy(L.copy())
    _poison_upper(Lt)
    assert torch.isnan(Lt[0, 3]) and torch.isinf(Lt[0, 1])
    mut, et, dgt = (torch.from_numpy(a) for a in (mu, eps, dg))
    assert rel_err(dense_fwd_ref(mut, Lt, et).numpy(), O.reparam(mu, L, eps, dense=True)) < 1e-13
    rdmu, rdL = O.reparam_dense_bwd(eps, dg)
    got = torch.cat([dense_bwd_ref_rows(et, dgt, r0, r1) for r0, r1 in _chunks(D)])
    assert rel_err(got.numpy(), rdL) < 1e-13
    v, _, rdL = O.kl_dense(mu, L, lam, grads=True)
    assert abs(kl_dense_ref(mut, Lt, lam) - v) < 1e-12 * abs(v)
    got = torch.cat([kl_dense_grad_ref_rows(Lt, lam, r0, r1) for r0, r1 in _chunks(D)])
    assert rel_err(got.numpy(), np.tril(rdL)) < 1e-13


# ------------------------------------------------------------------------------------------------- GPU helpers
def dev():
    return torch.device("cuda:0")


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan"), dtype=dtype, device=dev())


def _close(got, ref, what, tol):
    got = got.double().cpu().numpy() if isinstance(got, torch.Tensor) else got
    ref = ref.cpu().numpy() if isinstance(ref, torch.Tensor) else ref
    err = rel_err(got, ref)
    assert err <= tol, f"{what}: rel err {err:.3e} > {tol:g}"


def _stream():
    from whvi_b200 import functional as F
    return F._stream(dev())


def _lib():
    from whvi_b200 import _lib as lib
    return lib


@pytest.fixture(autouse=True)
def _free_device_memory():
    yield
    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _fwht_call(variant, x, out, scale=None):
    """One raw call of the variant's entry point; x, out: (rows, D) device tensors (out may be x)."""
    lib = _lib()
    L = lib.lib()
    rows, D = x.shape
    if variant == "scaled":
        rc = L.whvi_fwht_scaled_f32(x.data_ptr(), scale.data_ptr(), out.data_ptr(), rows, D, _stream())
    else:
        rc = getattr(L, f"whvi_fwht_{variant}")(x.data_ptr(), out.data_ptr(), rows, D, _stream())
    lib.check(rc, f"fwht {variant}")


def _fwht_id(case):
    return "-".join(str(c) for c in case)


# ------------------------------------------------------------------------------------------------- FWHT vs fp64
FWHT_TOL = 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("case", FWHT_SHAPES, ids=_fwht_id)
def test_fwht_vs_fp64(case):
    """fp32 and scaled against O.fwht (of x * s for scaled) at 1e-5, into NaN-filled outputs or in place; the scaled call
    equals the fp32 call on x * s bit for bit; the bf16 call equals bf16(fp32 call on the widened input) bit for bit."""
    from oracle import oracle as O
    variant, k, rows, inplace = case
    D = 1 << k
    gen = torch.Generator(device=dev()).manual_seed(k * 1000 + rows)
    x = torch.randn((rows, D), generator=gen, device=dev())
    if variant == "bf16":
        x = x.bfloat16()
    scale = torch.randn(D, generator=gen, device=dev()) if variant == "scaled" else None
    xin = (x.float() * scale) if variant == "scaled" else x.float()
    ref = O.fwht(xin.double().cpu().numpy())
    out = x.clone() if inplace else torch.full_like(x, float("nan"))
    _fwht_call(variant, out if inplace else x, out, scale)
    if variant == "bf16":
        y32 = _nan(rows, D)
        _fwht_call("f32", x.float(), y32)
        _close(y32, ref, f"fp32 call on the widened input {case}", FWHT_TOL)
        assert torch.equal(out, y32.bfloat16()), f"{case}: bf16 call is not bf16(fp32 call)"
    else:
        _close(out, ref, f"{case}", FWHT_TOL)
        if variant == "scaled":
            y32 = _nan(rows, D)
            _fwht_call("f32", xin, y32)
            assert torch.equal(out, y32), f"{case}: scaled call is not the transform of x * s"


@pytest.mark.gpu
@pytest.mark.parametrize("variant,k,rows", FWHT_LARGE, ids=[_fwht_id(c) for c in FWHT_LARGE])
def test_fwht_beyond_2_31_elements(variant, k, rows):
    """Calls of more than 2^31 elements (int64 indexing), every element compared chunk by chunk: fp32 against fwht_t in fp64
    on the device at 1e-5 of the chunk's largest; scaled equal to the fp32 call on x * s bit for bit; bf16 equal to
    bf16(fp32 call on the widened chunk) bit for bit, that fp32 call at 1e-5 of fp64."""
    D = 1 << k
    assert rows * D > 1 << 31
    gen = torch.Generator(device=dev()).manual_seed(rows + k)
    dt = torch.bfloat16 if variant == "bf16" else torch.float32
    x = torch.empty((rows, D), dtype=dt, device=dev())
    step = max(1, (1 << 27) // D)
    for r0 in range(0, rows, step):
        x[r0:r0 + step] = torch.randn((min(step, rows - r0), D), generator=gen, device=dev()).to(dt)
    scale = torch.randn(D, generator=gen, device=dev()) if variant == "scaled" else None
    out = torch.full_like(x, float("nan"))
    _fwht_call(variant, x, out, scale)
    for r0 in range(0, rows, step):
        r1 = min(rows, r0 + step)
        xc = x[r0:r1].float()
        if variant == "scaled":
            y32 = _nan(r1 - r0, D)
            _fwht_call("f32", xc * scale, y32)
            assert torch.equal(out[r0:r1], y32), f"rows {r0}:{r1}: scaled call is not the transform of x * s"
            continue
        ref = fwht_t(xc.double())
        if variant == "bf16":
            y32 = _nan(r1 - r0, D)
            _fwht_call("f32", xc, y32)
            assert torch.equal(out[r0:r1], y32.bfloat16()), f"rows {r0}:{r1}: bf16 call is not bf16(fp32 call)"
        else:
            y32 = out[r0:r1]
        err = float((y32.double() - ref).abs().max() / ref.abs().max())
        assert err <= FWHT_TOL, f"rows {r0}:{r1}: rel err {err:.3e}"
        del ref, y32


@pytest.mark.gpu
@pytest.mark.parametrize("k,rows,inplace", MULTIPASS_SHAPES)
def test_fwht_multipass_vs_fp64(k, rows, inplace):
    """D > 2^15: the persistent first pass over more than 148 segments, then passes of r = 1 .. 4 bits, as the only pass and
    as the tail, against fwht_t in fp64 on the device at 1e-5."""
    D = 1 << k
    gen = torch.Generator(device=dev()).manual_seed(k + rows)
    x = torch.randn((rows, D), generator=gen, device=dev())
    ref = fwht_t(x.double())
    out = x if inplace else torch.full_like(x, float("nan"))
    _fwht_call("f32", x, out)
    err = float((out.double() - ref).abs().max() / ref.abs().max())
    assert err <= FWHT_TOL, f"rel err {err:.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("k,rows", F64_SHAPES)
def test_fwht_f64_vs_oracle(k, rows):
    from oracle import oracle as O
    rng = np.random.default_rng(k * 100 + rows)
    x = rng.standard_normal((rows, 1 << k))
    xt = torch.from_numpy(x).to(dev())
    out = _nan(rows, 1 << k, dtype=torch.float64)
    lib = _lib()
    lib.check(lib.lib().whvi_fwht_f64(xt.data_ptr(), out.data_ptr(), rows, 1 << k, _stream()), "whvi_fwht_f64")
    _close(out, O.fwht(x), "fwht_f64", 1e-13)


# ------------------------------------------------------------------------------------------------- dense forward
DENSE_TOL = 1e-5
U32 = 2.0 ** -24   # unit roundoff of fp32


def gemm_tol(k_len):
    """Empirical bound on max|err| / max|ref| of a tcgen05 GEMM output whose TMEM accumulator takes a contraction of k_len:
    1e-5 up to k_len = 1024 (the lengths the earlier tests reach, where it holds); past that n u, with n = 3 k_len / 8
    accumulations (three tf32 MMAs per K = 8 step) and u the fp32 unit roundoff.  This is not a proven worst case: the error
    is measured against max|ref|, not against the largest partial sum.  It rests on measurements: the accumulator does not
    round to nearest, so on a B200 the error grows with k_len, not with its square root (2.2e-5 at k_len = 4096 and 7.9e-5 at
    16384 in the forward, 2.9e-5 at 4096 in dL, about a quarter of n u), while a skipped K block of 32 terms costs about
    1e-2."""
    return DENSE_TOL if k_len <= 1024 else 3 * (k_len // 8) * U32


def _dense_inputs(S, D, G, mu_stride, L_stride, seed):
    """mu (G, mu_stride), L (G, L_stride) with each block's (D, D) lower triangle at unit scale / sqrt(D) and NaN / inf above
    its diagonal (and in the stride padding), eps (G, S, D).  G = 0: one block, no padding."""
    Gn = max(G, 1)
    ms, ls = (mu_stride, L_stride) if G else (D, D * D)
    gen = torch.Generator(device=dev()).manual_seed(seed)
    mu = torch.randn((Gn, ms), generator=gen, device=dev())
    L = _nan(Gn, ls)
    for k in range(Gn):
        Lk = L[k, :D * D].view(D, D)
        for r0, r1 in _chunks(D):
            Lk[r0:r1] = torch.randn((r1 - r0, D), generator=gen, device=dev()) / np.sqrt(D)
        _poison_upper(Lk)
    eps = torch.randn((Gn, S, D), generator=gen, device=dev())
    return mu, L, eps


def _dense_fwd_call(mu, L, eps, S, D, G, mu_stride, L_stride, ws):
    lib = _lib()
    Lb = lib.lib()
    g = _nan(max(G, 1), S, D)
    if G == 0:
        rc = Lb.whvi_reparam_dense_f32(mu.data_ptr(), L.data_ptr(), eps.data_ptr(), g.data_ptr(), S, D, ws.data_ptr(),
                                       4 * ws.numel(), _stream())
    else:
        rc = Lb.whvi_reparam_dense_grouped_f32(mu.data_ptr(), mu_stride, L.data_ptr(), L_stride, eps.data_ptr(), g.data_ptr(), S,
                                               D, G, ws.data_ptr(), 4 * ws.numel(), _stream())
    lib.check(rc, "reparam_dense")
    return g


def _dense_fwd_id(case):
    S, D, G, *_ = case
    return f"S{S}-D{D}" + (f"-G{G}" if G else "")


@pytest.mark.gpu
@pytest.mark.parametrize("case", DENSE_FWD_SHAPES, ids=_dense_fwd_id)
def test_dense_forward_vs_fp64(case):
    """whvi_reparam_dense_f32 (G = 0) and whvi_reparam_dense_grouped_f32 into NaN-filled g with a NaN-filled workspace, L
    NaN / +-inf above the diagonal, against mu + eps @ tril(L)^T in fp64 at gemm_tol of a unit's contraction (1e-5 up to
    D = 8192).  Up to D = 8192 a second call with a
    workspace of random garbage gives the same bits."""
    from whvi_b200 import functional as F
    S, D, G, mu_stride, L_stride = case
    mu, L, eps = _dense_inputs(S, D, G, mu_stride, L_stride, S * 7 + D + G)
    name = "whvi_reparam_dense_grouped_workspace_bytes" if G else "whvi_reparam_dense_workspace_bytes"
    nbytes = F._query(name, S, D)[0]
    ws = _nan(_cdiv(nbytes, 4))
    g = _dense_fwd_call(mu, L, eps, S, D, G, mu_stride, L_stride, ws)
    tol = gemm_tol(min(dense_q(D), D // BM) * BM)   # a unit contracts over up to q column blocks
    for k in range(max(G, 1)):
        ref = dense_fwd_ref(mu[k, :D], L[k, :D * D].view(D, D), eps[k])
        err = float((g[k].double() - ref).abs().max() / ref.abs().max())
        assert err <= tol, f"block {k}: rel err {err:.3e} > {tol:.3e}"
        del ref
    if D <= 8192:
        ws.copy_(torch.randn(ws.shape, device=dev()) * 1e30)
        again = _dense_fwd_call(mu, L, eps, S, D, G, mu_stride, L_stride, ws)
        assert torch.equal(again, g), "not bit-reproducible with a garbage workspace"


# ------------------------------------------------------------------------------------------------- dense backward
def _dense_bwd_id(case):
    S, D, G = case
    return f"S{S}-D{D}-" + (f"G{G}" if G else "padded")


@pytest.mark.gpu
@pytest.mark.parametrize("case", DENSE_BWD_SHAPES, ids=_dense_bwd_id)
def test_dense_backward_vs_fp64(case):
    """G >= 1: whvi_reparam_dense_grouped_bwd_f32 (transpose, mode-1 GEMM, column sum) into NaN-filled dmu, dL and workspace;
    dL's upper triangle exactly 0.  G = 0: whvi_reparam_dense_bwd_f32 on caller-padded transposes into a NaN-filled dL: the
    lower triangle against fp64, the diagonal tiles' upper part exactly 0, the tiles above them not written (still NaN).
    dL = tril(dg^T eps) within sum_err gemm_tol(Sp) and dmu = sum_s dg within sum_err 1e-5 of fp64."""
    from whvi_b200 import functional as F
    S, D, G = case
    lib = _lib()
    Gn = max(G, 1)
    gen = torch.Generator(device=dev()).manual_seed(S + D + G)
    eps = torch.randn((Gn, S, D), generator=gen, device=dev())
    dg = torch.randn((Gn, S, D), generator=gen, device=dev())
    dL = _nan(Gn, D, D)
    dmu = _nan(Gn, D)
    if G:
        nbytes = F._query("whvi_reparam_dense_grouped_workspace_bytes", S, D)[0]
        ws = _nan(_cdiv(nbytes, 4))
        lib.check(lib.lib().whvi_reparam_dense_grouped_bwd_f32(eps.data_ptr(), dg.data_ptr(), dmu.data_ptr(), dL.data_ptr(), S, D,
                                                               G, ws.data_ptr(), nbytes, _stream()), "reparam_dense_grouped_bwd")
        del ws
    else:
        Sp = _round_up(S, BK)
        dgT, eT = torch.zeros((D, Sp), device=dev()), torch.zeros((D, Sp), device=dev())
        dgT[:, :S] = dg[0].T
        eT[:, :S] = eps[0].T
        lib.check(lib.lib().whvi_reparam_dense_bwd_f32(dgT.data_ptr(), eT.data_ptr(), dL.data_ptr(), Sp, D, _stream()),
                  "reparam_dense_bwd")
    for k in range(Gn):
        if G:
            assert sum_err(dmu[k], dg[k].double().sum(0), S) <= DENSE_TOL, f"dmu block {k}"
        err = ref_max = 0.0
        for r0, r1 in _chunks(D):
            ref = dense_bwd_ref_rows(eps[k], dg[k], r0, r1)
            got = dL[k, r0:r1]
            up = _upper(r0, r1, D, dev())
            if G:
                assert torch.count_nonzero(torch.where(up, got, 0.0)) == 0, f"block {k} rows {r0}:{r1}: upper triangle not 0"
            else:
                tile_up = torch.arange(D, device=dev())[None, :] // BM > torch.arange(r0, r1, device=dev())[:, None] // BM
                assert bool(torch.isnan(got[tile_up]).all()), f"rows {r0}:{r1}: a tile above the diagonal was written"
                assert torch.count_nonzero(got[up & ~tile_up]) == 0, f"rows {r0}:{r1}: diagonal tile not 0 above the diagonal"
                got = torch.where(tile_up, 0.0, got)
            assert bool(torch.isfinite(got).all()), f"block {k} rows {r0}:{r1}: dL not finite on or below the diagonal"
            err = _worst(err, float((got.double() - ref).abs().max()))
            ref_max = _worst(ref_max, float(ref.abs().max()))
        tol = gemm_tol(_round_up(S, BK))
        assert err / max(ref_max, np.sqrt(S)) <= tol, f"dL block {k}: sum err {err / max(ref_max, np.sqrt(S)):.3e} > {tol:.3e}"


# ------------------------------------------------------------------------------------------------- small D
@pytest.mark.gpu
@pytest.mark.parametrize("S,D,G,mu_stride,L_stride", SMALL_SHAPES)
def test_small_d_vs_oracle(S, D, G, mu_stride, L_stride):
    """reparam_dense_small_kernel and reparam_dense_small_bwd_kernel through the grouped entry points, NaN-filled outputs and
    L NaN / inf above the diagonal and in the stride padding, against O.reparam(dense=True) and O.reparam_dense_bwd within
    sum_err 1e-5 (fp32 chains of D and S terms); dL exactly 0 above the diagonal; a second call gives the same bits."""
    from oracle import oracle as O
    lib = _lib()
    Lb = lib.lib()
    mu, L, eps = _dense_inputs(S, D, G, mu_stride, L_stride, S + D * 10 + G)
    gen = torch.Generator(device=dev()).manual_seed(S * 3 + D)
    dg = torch.randn((G, S, D), generator=gen, device=dev())

    def run():
        g, dmu, dL = _nan(G, S, D), _nan(G, D), _nan(G, D, D)
        lib.check(Lb.whvi_reparam_dense_grouped_f32(mu.data_ptr(), mu_stride, L.data_ptr(), L_stride, eps.data_ptr(), g.data_ptr(),
                                                    S, D, G, None, 0, _stream()), "reparam_dense_grouped (small D)")
        lib.check(Lb.whvi_reparam_dense_grouped_bwd_f32(eps.data_ptr(), dg.data_ptr(), dmu.data_ptr(), dL.data_ptr(), S, D, G,
                                                        None, 0, _stream()), "reparam_dense_grouped_bwd (small D)")
        return g, dmu, dL

    g, dmu, dL = run()
    mu64, L64, e64, dg64 = (a.double().cpu().numpy() for a in (mu, L, eps, dg))
    for k in range(G):
        Lk = np.tril(np.nan_to_num(L64[k, :D * D].reshape(D, D), nan=0.0, posinf=0.0, neginf=0.0))
        ref = O.reparam(mu64[k, :D], Lk, e64[k], dense=True)
        assert sum_err(g[k].cpu(), torch.from_numpy(ref), D) <= DENSE_TOL, f"g block {k}"
        rdmu, rdL = O.reparam_dense_bwd(e64[k], dg64[k])
        assert sum_err(dmu[k].cpu(), torch.from_numpy(rdmu), S) <= DENSE_TOL, f"dmu block {k}"
        assert sum_err(dL[k].cpu(), torch.from_numpy(rdL), S) <= DENSE_TOL, f"dL block {k}"
        assert torch.count_nonzero(torch.triu(dL[k], 1)) == 0
    again = run()
    assert all(torch.equal(a, b) for a, b in zip(again, (g, dmu, dL)))


# ------------------------------------------------------------------------------------------------- dense KL
def _kl_id(case):
    D, G, *_, gs = case
    return f"D{D}-" + (f"G{G}" if G else "plain") + f"-gs{gs}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", KL_DENSE_SHAPES, ids=_kl_id)
def test_kl_dense_vs_fp64(case):
    """whvi_kl_dense_f32 (G = 0) and whvi_kl_dense_grouped_f32, L positive on the diagonal and NaN / inf above it, into a
    NaN-filled scalar, dmu, dL and workspace: the value against the sum of the per-block O.kl_dense (kl_dense_ref at
    D = 16384) to 1e-5, dmu and dL (times grad_scale) at 1e-5, dL exactly 0 above the diagonal."""
    from oracle import oracle as O
    D, G, mu_stride, L_stride, gs = case
    lib = _lib()
    lam = 0.3
    Gn = max(G, 1)
    mu, L, _ = _dense_inputs(0, D, G, mu_stride, L_stride, D + G)
    for k in range(Gn):
        diag = L[k, :D * D].view(D, D).diagonal()
        diag.copy_(diag.abs() + 0.05)
    out, dmu, dL, ws = _nan(1), _nan(Gn, D), _nan(Gn, D, D), _nan(2 * Gn * D)
    if G:
        rc = lib.lib().whvi_kl_dense_grouped_f32(mu.data_ptr(), mu_stride, L.data_ptr(), L_stride, lam, D, G, out.data_ptr(),
                                                 dmu.data_ptr(), dL.data_ptr(), gs, ws.data_ptr(), 4 * ws.numel(), _stream())
    else:
        rc = lib.lib().whvi_kl_dense_f32(mu.data_ptr(), L.data_ptr(), lam, D, out.data_ptr(), dmu.data_ptr(), dL.data_ptr(), gs,
                                         ws.data_ptr(), 4 * ws.numel(), _stream())
    lib.check(rc, "kl_dense")
    value = 0.0
    for k in range(Gn):
        muk, Lk = mu[k, :D], L[k, :D * D].view(D, D)
        if D >= 16384:
            value += kl_dense_ref(muk, Lk, lam)
            err = ref_max = 0.0
            for r0, r1 in _chunks(D):
                ref = gs * kl_dense_grad_ref_rows(Lk, lam, r0, r1)
                assert bool(torch.isfinite(dL[k, r0:r1]).all()), f"dL rows {r0}:{r1} not finite"
                err = _worst(err, float((dL[k, r0:r1].double() - ref).abs().max()))
                ref_max = _worst(ref_max, float(ref.abs().max()))
                assert torch.count_nonzero(torch.where(_upper(r0, r1, D, dev()), dL[k, r0:r1], 0.0)) == 0
            assert err <= DENSE_TOL * ref_max, f"dL: rel err {err / ref_max:.3e}"
            _close(dmu[k], gs * muk.double() / lam, "dmu", DENSE_TOL)
        else:
            L64 = np.tril(np.nan_to_num(Lk.double().cpu().numpy(), nan=0.0, posinf=0.0, neginf=0.0))
            v, rdmu, rdL = O.kl_dense(muk.double().cpu().numpy(), L64, lam, grads=True)
            value += v
            _close(dmu[k], gs * rdmu, f"dmu block {k}", DENSE_TOL)
            _close(dL[k], gs * np.tril(rdL), f"dL block {k}", DENSE_TOL)
            assert torch.count_nonzero(torch.triu(dL[k], 1)) == 0
    assert abs(out.item() - value) <= DENSE_TOL * abs(value), (out.item(), value)


# ------------------------------------------------------------------------------------------------- MC moments
@pytest.mark.gpu
@pytest.mark.parametrize("S,n,stride,accumulate", MC_MOMENTS_SHAPES)
def test_mc_moments_vs_fp64(S, n, stride, accumulate):
    """whvi_mc_moments_strided_f32: out = in + sum_s y and in2 + sum_s y^2 (samples at a stride >= n) into NaN-filled outputs,
    against fp64 within sum_err 1e-6 (the samples' 4-wide loop and its tail, a partly idle last CTA)."""
    lib = _lib()
    gen = torch.Generator(device=dev()).manual_seed(S + n)
    y = torch.randn((S, stride), generator=gen, device=dev())
    y[:, n:] = float("nan")   # past n in every sample: never read
    a0 = torch.randn(n, generator=gen, device=dev()) if accumulate else None
    b0 = torch.randn(n, generator=gen, device=dev()) if accumulate else None
    oa, ob = _nan(n), _nan(n)
    lib.check(lib.lib().whvi_mc_moments_strided_f32(y.data_ptr(), stride, a0.data_ptr() if accumulate else None,
                                                    b0.data_ptr() if accumulate else None, oa.data_ptr(), ob.data_ptr(), S, n,
                                                    _stream()), "mc_moments_strided")
    y64 = y[:, :n].double()
    ra, rb = y64.sum(0), (y64 * y64).sum(0)
    if accumulate:
        ra, rb = ra + a0.double(), rb + b0.double()
    assert sum_err(oa, ra, S + 1) <= 1e-6
    assert sum_err(ob, rb, S + 1) <= 1e-6
