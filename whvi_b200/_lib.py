"""Binding of libwhvi_b200.so (C ABI declared in include/whvi_b200.h): ctypes loads the library and declares every
signature; the launch calls whose parameters are all pointers / integers are then handed out behind a small CPython shim
(csrc_host/fastcall.c) that calls the same function without ctypes' per-call marshalling.

There is no fallback of any kind: if the library is missing or a call fails, a
RuntimeError is raised (mirroring the TORCH_CHECK -> RuntimeError behaviour of the
reference extension, src/fwht/cuda/fwht_cuda.cpp:6-10).
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_float, c_int, c_int64, c_size_t, c_void_p
from pathlib import Path

import os

# WHVI_B200_LIB=/path/to/libwhvi_b200_NAME.so loads an A/B variant build (python -m whvi_b200.build
# --variant NAME -D...) in place of the product library, so the whole test-suite and bench.py can be
# run against it.  Same C ABI, still no fallback of any kind.
LIB_PATH = Path(os.environ.get("WHVI_B200_LIB") or Path(__file__).resolve().parent / "libwhvi_b200.so")

# name -> (restype, argtypes); kept in one place so tests can check that every symbol
# the header declares is exported and bound.
FP = POINTER(c_float)
SIGNATURES = {
    "whvi_abi_version": (c_int, []),
    "whvi_last_error": (c_char_p, []),
    "whvi_max_dim": (c_int64, []),
    "whvi_fwht_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "whvi_layer_fwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int64, c_int64, c_int64, c_void_p]),
    "whvi_layer_bwd_workspace_bytes": (c_int, [c_int64, c_int64, c_int64, POINTER(c_size_t)]),
    "whvi_layer_bwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64,
                                   c_void_p]),
    "whvi_layer_fwd_partials": (c_int, [c_int64, c_int64, c_int64, POINTER(c_int64)]),
    "whvi_layer_fwd_fused_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "whvi_layer_bwd_fused_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64,
                                         c_int, c_void_p, c_void_p, c_void_p]),
    "whvi_layer_bwd_scaled_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64,
                                          c_int64, c_int, c_void_p]),
    "whvi_layer_loss_sizes": (c_int, [c_int64, c_int64, c_int64, POINTER(c_size_t), POINTER(c_int64)]),
    "whvi_layer_loss_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64,
                                    c_int64, c_int64, c_int, c_void_p]),
    "whvi_reparam_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p]),
    "whvi_reparam_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int,
                                     c_void_p]),
    "whvi_reparam_dense_workspace_bytes": (c_int, [c_int64, c_int64, POINTER(c_size_t)]),
    "whvi_reparam_dense_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_size_t, c_void_p]),
    "whvi_reparam_dense_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "whvi_kl_dense_f32": (c_int, [c_void_p, c_void_p, c_float, c_int64, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_size_t,
                                  c_void_p]),
    "whvi_reparam_dense_grouped_workspace_bytes": (c_int, [c_int64, c_int64, POINTER(c_size_t)]),
    "whvi_reparam_dense_grouped_f32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                               c_void_p, c_size_t, c_void_p]),
    "whvi_reparam_dense_grouped_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p, c_size_t,
                                                   c_void_p]),
    "whvi_kl_dense_grouped_f32": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_float, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                                          c_float, c_void_p, c_size_t, c_void_p]),
    "whvi_stacked_fwd_g_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                       c_int64, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_stacked_bwd_g_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int64, c_int64, c_int,
                                       c_void_p]),
    "whvi_column_fwd_g_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                      c_int64, c_int64, c_int, c_int, c_void_p]),
    "whvi_column_bwd_g_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "whvi_pad_rows_f32": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "whvi_stacked_fwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_stacked_bwd_workspace_bytes": (c_int, [c_int64, c_int64, c_int64, c_int64, c_int, POINTER(c_size_t)]),
    "whvi_stacked_bwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                     c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64,
                                     c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_column_fwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "whvi_column_bwd_workspace_bytes": (c_int, [c_int64, c_int64, c_int64, POINTER(c_size_t)]),
    "whvi_column_bwd_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int64,
                                    c_int, c_int, c_void_p]),
    "whvi_kl_grouped_f32": (c_int, [c_void_p, c_void_p, c_float, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p,
                                    c_float, c_void_p]),
    "whvi_layer_moments_add_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_fwht_scaled_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "whvi_fwht_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "whvi_layer_fwd_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                    c_int, c_void_p]),
    "whvi_layer_bwd_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_layer_loss_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int,
                                     c_void_p]),
    # bf16 twins of the Stacked and Column calls: the fp32 signatures with void* activations
    "whvi_pad_rows_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "whvi_stacked_fwd_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_stacked_fwd_g_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                        c_int64, c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_stacked_bwd_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                      c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64,
                                      c_int64, c_int64, c_int64, c_int, c_void_p]),
    "whvi_stacked_bwd_g_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int64, c_int64, c_int,
                                        c_void_p]),
    "whvi_column_fwd_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_int64, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "whvi_column_fwd_g_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                       c_int64, c_int64, c_int, c_int, c_void_p]),
    "whvi_column_bwd_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int64,
                                     c_int, c_int, c_void_p]),
    "whvi_column_bwd_g_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_int64, c_int, c_int, c_void_p]),
    "whvi_fwht_f64": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "whvi_mc_moments_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p]),
    "whvi_mc_moments_strided_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                            c_void_p]),
    "whvi_layer_moments_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                       c_int64, c_int64, c_int, c_void_p]),
    "whvi_adam_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_void_p, c_void_p, c_float,
                              c_float, c_float, c_float, c_void_p]),
    "whvi_kl_f32": (c_int, [c_void_p, c_void_p, c_float, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_float, c_int,
                            c_void_p]),
    # categorical likelihood: the _bf16 twins have the fp32 signatures with void* logits / dz
    "whvi_categorical_sizes": (c_int, [c_int64, c_int64, POINTER(c_size_t)]),
    "whvi_categorical_nll_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_void_p]),
    "whvi_categorical_nll_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64, c_void_p]),
    "whvi_categorical_nll_bwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    "whvi_categorical_nll_bwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p]),
    # the _ex calls: the plain arguments, then weight, label_smoothing (float: stays on ctypes), ignore_index and flags
    "whvi_categorical_nll_ex_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64,
                                            c_void_p, c_float, c_int64, c_int, c_void_p]),
    "whvi_categorical_nll_ex_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_int64, c_int64, c_int64,
                                             c_void_p, c_float, c_int64, c_int, c_void_p]),
    "whvi_categorical_nll_bwd_ex_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                                c_float, c_int64, c_int, c_void_p]),
    "whvi_categorical_nll_bwd_ex_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_void_p,
                                                 c_float, c_int64, c_int, c_void_p]),
    "whvi_categorical_predictive_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int,
                                                c_void_p]),
    "whvi_categorical_predictive_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int,
                                                 c_void_p]),
    "whvi_categorical_uncertainty_f32": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                                 c_int64, c_int, c_void_p]),
    "whvi_categorical_uncertainty_bf16": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64,
                                                  c_int64, c_int, c_void_p]),
    # convolution patches: geometry (S, B, H, W, C, kh, kw, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w) as int64
    "whvi_im2col_f32": (c_int, [c_void_p, c_int64, c_void_p] + [c_int64] * 14 + [c_void_p]),
    "whvi_im2col_bf16": (c_int, [c_void_p, c_int64, c_void_p] + [c_int64] * 14 + [c_void_p]),
    "whvi_col2im_f32": (c_int, [c_void_p, c_int64, c_void_p] + [c_int64] * 13 + [c_int, c_void_p]),
    "whvi_col2im_bf16": (c_int, [c_void_p, c_int64, c_void_p] + [c_int64] * 13 + [c_int, c_void_p]),
}

_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m whvi_b200.build` "
                "(whvi_b200 has no CPU or PyTorch fallback)")
        L = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.whvi_abi_version() != 1:
            raise RuntimeError("libwhvi_b200.so ABI version mismatch; rebuild with python -m whvi_b200.build --force")
        _lib = _FastLib(L)
    return _lib


class _FastLib:
    """The loaded library.  Attribute access gives the entry point as a callable; for entry points whose parameters are all
    pointers / integers (every launch call of the hot path) that callable goes through the CPython shim ``_fastcall.calli``
    (``csrc_host/fastcall.c``) instead of ctypes' per-call argument marshalling: the same C-ABI function, the same arguments,
    ~3 us less host time per call (measured on the published per-call FWHT benchmark: 9.5 -> 5.9 us).  Entry points with
    ``float`` or output-pointer parameters, and everything when the shim is not built, stay on ctypes."""

    _INT_TYPES = (c_void_p, c_int64, c_int, c_size_t)

    def __init__(self, cdll):
        self._cdll = cdll
        try:
            from . import _fastcall
        except Exception:
            _fastcall = None
        self._fc = _fastcall

    def __getattr__(self, name):
        fn = getattr(self._cdll, name)
        sig = SIGNATURES.get(name)
        if (self._fc is not None and sig is not None and sig[0] is c_int and 4 <= len(sig[1]) <= 25
                and all(t in self._INT_TYPES for t in sig[1])):
            import functools
            fn = functools.partial(self._fc.calli, ctypes.cast(fn, c_void_p).value)
        setattr(self, name, fn)   # next access is a plain attribute hit
        return fn


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().whvi_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed ({rc}): {msg}")
