"""CPU: the C-ABI library loads, exports every symbol include/whvi_b200.h declares, and
the Python frontends reject bad input the way the reference's TORCH_CHECKs do.  No
compute call is made (there is no GPU here)."""
import ctypes
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def declared_symbols():
    text = (ROOT / "include" / "whvi_b200.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"WHVI_API\s+[\w\s\*]+?\b(whvi_\w+)\s*\(", text)))


def test_header_declares_something():
    syms = declared_symbols()
    assert "whvi_fwht_f32" in syms and "whvi_last_error" in syms


def test_library_exports_every_declared_symbol():
    from whvi_b200 import _lib
    L = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in declared_symbols():
        assert hasattr(L, name), f"{name} declared in include/whvi_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in whvi_b200/_lib.py"
    assert _lib.lib().whvi_abi_version() == 1
    assert _lib.lib().whvi_max_dim() >= 1 << 20


def test_fwht_frontend_rejects_like_the_reference():
    from whvi_b200 import FWHTFunction
    with pytest.raises(RuntimeError, match="X must be a CUDA tensor"):
        FWHTFunction.apply(torch.randn(2, 4))


def test_no_oracle_import_in_product():
    """The product path must never route through oracle/ (or /root/reference)."""
    for py in (ROOT / "whvi_b200").rglob("*.py"):
        src = py.read_text()
        assert "oracle" not in src.replace("# oracle", ""), f"{py} mentions the oracle"
        assert "/root/reference" not in src


def test_argument_validation_without_a_gpu():
    """Every entry point validates its arguments before it touches CUDA: bad calls return a negative
    WHVI_E_* code and leave a message in whvi_last_error() (what the Python side turns into the
    RuntimeError the reference's TORCH_CHECKs raise, src/fwht/cuda/fwht_cuda.cpp:6-10).  No kernel runs."""
    from whvi_b200 import _lib
    L = _lib.lib()
    a = 1 << 20        # a 16-byte aligned fake "device pointer" that is never dereferenced
    E_NULL, E_SHAPE, E_ALIGN, E_MODE = -1, -2, -3, -4

    def err():
        return L.whvi_last_error().decode()

    assert L.whvi_fwht_f32(a, a, 4, 12, None) == E_SHAPE and "power of 2" in err()         # fwht_cuda.cpp:10
    assert L.whvi_fwht_f32(a, a, -1, 16, None) == E_SHAPE
    assert L.whvi_fwht_f32(None, a, 4, 16, None) == E_NULL
    assert L.whvi_fwht_f32(a + 4, a, 4, 16, None) == E_ALIGN
    assert L.whvi_fwht_f32(a, a, 0, 16, None) == 0                                         # empty batch: no-op
    assert L.whvi_fwht_f64(a, a, 4, 24, None) == E_SHAPE
    # fused layer: D range, power of two, sample stride, flags, pointers
    assert L.whvi_layer_fwd_f32(a, 0, a, a, a, None, a, 2, 3, 48, None) == E_SHAPE
    assert L.whvi_layer_fwd_f32(a, 0, a, a, a, None, a, 2, 3, 2, None) == E_SHAPE and "outside" in err()
    assert L.whvi_layer_fwd_f32(a, 7, a, a, a, None, a, 2, 3, 64, None) == E_SHAPE and "x_sample_stride" in err()
    assert L.whvi_layer_fwd_f32(None, 0, a, a, a, None, a, 2, 3, 64, None) == E_NULL
    assert L.whvi_layer_fwd_fused_f32(a, 0, a, a, a, None, a, 2, 3, 64, 8, None, None, None) == E_MODE
    assert L.whvi_layer_fwd_fused_f32(a, 0, a, a, a, None, a, 2, 3, 64, 0, a, None, None) == E_NULL  # target without partials
    assert L.whvi_layer_fwd_f32(a, 0, a, a, a, None, a, 0, 3, 64, None) == 0                # S = 0: nothing to do
    ws = ctypes.c_size_t(0)
    assert L.whvi_layer_bwd_workspace_bytes(2, 3, 1 << 14, ctypes.byref(ws)) == E_SHAPE     # backward stops at 8192
    assert L.whvi_layer_bwd_workspace_bytes(16, 4096, 4096, ctypes.byref(ws)) == 0 and ws.value > 0
    assert L.whvi_layer_bwd_f32(a, 0, a, a, a, a, a, None, a, a, None, a, 0, 2, 3, 64, None) == E_NULL   # dg missing
    assert L.whvi_layer_bwd_f32(a, 0, a, a, a, a, a, a, a, a, None, a, 16, 2, 3, 64, None) == -5          # workspace too small
    n_sq = ctypes.c_int64(0)
    assert L.whvi_layer_loss_sizes(2, 3, 64, ctypes.byref(ws), ctypes.byref(n_sq)) in (0, E_SHAPE)
    assert L.whvi_reparam_f32(a, a, a, a, 2, 64, 7, None) == E_MODE
    assert L.whvi_kl_f32(a, a, ctypes.c_float(-1.0), 64, 0, a, None, None, ctypes.c_float(1.0), 0, None) == E_SHAPE
    assert L.whvi_kl_f32(a, a, ctypes.c_float(1.0), 64, 5, a, None, None, ctypes.c_float(1.0), 0, None) == E_MODE
    assert L.whvi_mc_moments_f32(a, a, a, 2, 6, 0, None) == E_SHAPE                          # n % 4
    assert L.whvi_mc_moments_strided_f32(a, 8, None, None, a, None, 2, 16, None) == E_SHAPE  # stride < n
    assert L.whvi_mc_moments_f32(a, None, a, 2, 8, 0, None) == E_NULL


def test_stacked_rejects_more_than_65535_groups_without_a_gpu():
    """G > 65535 would be the grouped reparameterisation backward's grid.y: every Stacked entry point rejects it with
    WHVI_E_SHAPE before any CUDA call (null pointers: the shape check comes first)."""
    from whvi_b200 import _lib
    L = _lib.lib()
    E_SHAPE = -2
    G, D, S, B = 65536, 4, 1, 1
    ws = ctypes.c_size_t(0)
    assert L.whvi_stacked_bwd_workspace_bytes(S, B, D, G, 0, ctypes.byref(ws)) == E_SHAPE
    assert b"above 65535" in L.whvi_last_error()
    assert L.whvi_stacked_fwd_f32(None, 0, None, None, None, None, D, None, None, None, None, None, S, B, D, G, G * D, 0,
                                  None) == E_SHAPE
    assert L.whvi_stacked_bwd_f32(None, 0, None, None, None, None, None, D, None, None, D, None, None, None, None, None, None, 0,
                                  S, B, D, G, G * D, 0, None) == E_SHAPE
    assert b"above 65535" in L.whvi_last_error()
    assert L.whvi_stacked_bwd_workspace_bytes(S, B, D, 65535, 0, ctypes.byref(ws)) == 0   # the limit itself is fine


def test_shim_and_ctypes_reach_the_same_entry_points():
    """The CPython shim (csrc_host/fastcall.c) is a second way INTO the C ABI, not around it: for the all-integer entry points
    it hands out, the status codes and error messages equal what the ctypes binding of the same function returns (argument
    validation only -- no GPU is touched), new entry points of this round included."""
    from whvi_b200 import _lib
    L = _lib.lib()
    raw = L._cdll
    if L._fc is None:
        pytest.skip("the shim is optional; ctypes is the binding without it")
    a = 1 << 20   # a fake, 16-byte aligned "device pointer": validation failures come before any dereference
    cases = [
        ("whvi_fwht_f32", (a, a, 4, 12, None)),
        ("whvi_fwht_f32", (a + 4, a, 4, 16, None)),
        ("whvi_fwht_bf16", (a, a, 4, 24, None)),
        ("whvi_fwht_scaled_f32", (a, None, a, 4, 16, None)),
        ("whvi_layer_fwd_f32", (a, 7, a, a, a, None, a, 2, 3, 64, None)),
        ("whvi_layer_fwd_bf16", (a, 0, a, a, a, None, a, 2, 3, 48, 0, None)),
        ("whvi_layer_bwd_f32", (a, 0, a, a, a, a, a, a, a, a, None, a, 16, 2, 3, 64, None)),
        ("whvi_stacked_fwd_f32", (a, 0, a, a, a, a, 8, a, None, a, a, a, 2, 3, 16, 4, 64, 0, None)),       # param_stride < D
        ("whvi_stacked_fwd_f32", (a, 0, a, a, a, a, 16, a, None, a, a, a, 2, 3, 16, 4, 100, 0, None)),     # n_out does not match G * D
        ("whvi_stacked_bwd_f32", (a, 0, a, a, a, a, a, 16, a, None, 13, None, a, a, a, None, a, 0, 2, 3, 16, 4, 64, 0, None)),
        ("whvi_column_fwd_f32", (a, 0, a, a, a, a, a, None, a, a, a, 2, 3, 16, 5, 1, 0, None)),            # D != next_pow2(n)
        ("whvi_column_bwd_f32", (a, 0, a, a, a, a, a, a, None, a, a, a, a, None, a, 0, 2, 3, 16, 16, 0, 1, None)),  # RELU_IN on the plain form
        ("whvi_layer_moments_add_f32", (a, 0, a, a, a, None, a + 4, None, a, a, 2, 3, 8192, 0, None)),
        ("whvi_pad_rows_f32", (a, a, 3, 20, 16, None)),
        ("whvi_mc_moments_f32", (a, a, a, 2, 6, 0, None)),
    ]
    for name, args in cases:
        fast = getattr(L, name)
        assert not hasattr(fast, "argtypes"), name          # handed out behind the shim
        rc_fast, msg_fast = fast(*args), L.whvi_last_error()
        rc_raw, msg_raw = getattr(raw, name)(*args), L.whvi_last_error()
        assert rc_fast == rc_raw and rc_fast < 0, (name, rc_fast, rc_raw)
        assert msg_fast == msg_raw and msg_fast, name
    # float or output-pointer parameters stay on ctypes
    assert hasattr(L.whvi_kl_f32, "argtypes") and hasattr(L.whvi_layer_bwd_workspace_bytes, "argtypes")
