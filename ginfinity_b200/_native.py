"""ctypes binding of libgfx.so (the C ABI declared in include/gfx.h).

There is no fallback: if the library is missing, importing this module
raises, and every encoder entry point fails loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

import os

# GFX_LIBRARY: developer override (A/B runs of two builds on the same board)
_LIB_PATH = Path(os.environ.get("GFX_LIBRARY") or Path(__file__).resolve().parent / "libgfx.so")

GFX_F16, GFX_F32 = 0, 1
IMPL_AUTO, IMPL_SIMT, IMPL_UMMA, IMPL_UMMA_LEAN, IMPL_SPLIT = 0, 1, 2, 5, 8


class NativeError(RuntimeError):
    """A libgfx call returned a non-zero status."""


class NativeLibraryMissing(ImportError):
    pass


if not _LIB_PATH.is_file():
    raise NativeLibraryMissing(
        f"{_LIB_PATH} has not been built; run `python -m "
        "ginfinity_b200.build_native` (needs nvcc). ginfinity_b200 has no "
        "CPU or eager fallback.")

lib = C.CDLL(str(_LIB_PATH))

_p, _i32, _i64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t


class FoldedWeightsStruct(C.Structure):
    _fields_ = [("hidden", _i32), ("layers", _i32), ("out_dim", _i32),
                ("feature_dim", _i32), ("edge_dim", _i32)] + [
        (name, _p) for name in (
            "w_in", "b_in", "table", "eps1", "w1", "b1", "w2", "b2",
            "ln_g", "ln_b", "wa", "ba", "wb", "bb")]


_SIGNATURES = {
    "gfx_abi_version": (C.c_int, []),
    "gfx_last_error": (C.c_char_p, []),
    "gfx_model_create": (C.c_int, [C.POINTER(FoldedWeightsStruct), C.POINTER(_p)]),
    "gfx_model_destroy": (C.c_int, [_p]),
    "gfx_pack_microbatches": (C.c_int, [_p, _p, _i64, _i64, _i64, _p, _p, _p, _p]),
    "gfx_csr_workspace_bytes": (_sz, [_i64, _i64]),
    "gfx_csr_build": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _sz, _p]),
    "gfx_csr_build_checked": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _p, _sz, _p]),
    "gfx_edge_describe_workspace_bytes": (_sz, [_i64]),
    "gfx_edge_describe": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _p, _p, _p, _sz, _p]),
    "gfx_csr_build_if": (C.c_int, [_p, _p, _p, _i64, _i64, _i32, _p, _p, _p, _p, _p, _sz, _p]),
    "gfx_graph_workspace_bytes": (_sz, [_i64, _i64]),
    "gfx_graph_count": (C.c_int, [_p, _p, _i64, _i64, C.c_int, _p, _p, _p, _sz, _p]),
    "gfx_graph_fill": (C.c_int, [_p, _p, _p, _p, _i64, _i64, _i64, C.c_int, _p, _p, _p, _p, _p,
                                 _p, _p, _p, _p, _sz, _p]),
    "gfx_slice_workspace_bytes": (_sz, [_i64, _i64]),
    "gfx_slice_select": (C.c_int, [_p, _p, _p, _p, _i64, _i64, C.c_int, C.c_int, C.c_int, _p, _p,
                                   _p, _p, _sz, _p]),
    "gfx_slice_fill": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _i64, _i64, _i64, C.c_int, _p,
                                 _p, _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gfx_core_rows_workspace_bytes": (_sz, [_i64]),
    "gfx_core_rows": (C.c_int, [_p, _i64, _p, _p, _p, _sz, _p]),
    "gfx_input_linear": (C.c_int, [_p, _p, _i64, _p, C.c_int, _p]),
    "gfx_aggregate": (C.c_int, [_p, C.c_int, _p, _p, _p, _p, _i64, _p, C.c_int, _p]),
    "gfx_aggregate_banded": (C.c_int, [_p, C.c_int, _p, _p, _p, _p, _p, _p, _i64, _p, C.c_int, _p]),
    "gfx_mlp_ln_residual": (C.c_int, [_p, C.c_int, _p, _p, _i64, _p, C.c_int, C.c_int, _p]),
    "gfx_layer_fused_pair": (C.c_int, [_p, C.c_int, _p, _p, _p, _p, _i64, _p, _p]),
    "gfx_row_describe": (C.c_int, [_p, _p, _p, _i64, _p, _p]),
    "gfx_layer_fused_banded": (C.c_int, [_p, C.c_int, _p, _p, _p, _p, _p, _i64, _p, _p]),
    "gfx_head_l2norm": (C.c_int, [_p, _p, _p, _i64, _p, C.c_int, C.c_int, C.c_int, _p]),
    "gfx_encode_workspace_bytes": (_sz, [_i64, C.c_int]),
    "gfx_encode": (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _p, C.c_int, C.c_int,
                             C.c_int, C.c_int, _p, _sz, _p]),
    "gfx_encode_described": (C.c_int, [_p, _p, _p, _p, _p, _p, _i64, _p, C.c_int, _p, _sz, _p]),
    "gfx_encode_described_f32": (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i64, _p, C.c_int, _p, _sz,
                                           _p]),
    "gfx_topk_workspace_bytes": (_sz, [_i64, _i64, C.c_int]),
    "gfx_topk": (C.c_int, [_p, _i64, _p, _i64, C.c_int, C.c_int, C.c_int, _i64,
                           _p, _p, _p, _sz, _p]),
    "gfx_topk_f32_prepare": (C.c_int, [_p, _i64, _p, _p]),
    "gfx_topk_f32_workspace_bytes": (_sz, [_i64, _i64, C.c_int]),
    "gfx_topk_f32": (C.c_int, [_p, _i64, _p, _p, _i64, C.c_int, C.c_int, C.c_int, _i64,
                               _p, _p, _p, _sz, _p]),
    "gfx_topk_merge": (C.c_int, [_p, _p, C.c_int, _i64, C.c_int, _p, _p, _p]),
    "gfx_align_workspace_bytes": (_sz, [_i64, _i64]),
    "gfx_align": (C.c_int, [_p, _i64, _p, _i64, _p, _i64, C.c_float, C.c_float, C.c_float,
                            _p, _p, _p, _sz, _p]),
    "gfx_align_trace_workspace_bytes": (_sz, [_i64, _i64]),
    "gfx_align_trace": (C.c_int, [_p, _i64, _p, _i64, _p, _i64, C.c_float, C.c_float, C.c_float,
                                  _p, _p, _p, _p, _p, _p, _sz, _p]),
    "gfx_profile_enable": (C.c_int, [C.c_uint32]),
    "gfx_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(_i64), C.c_int]),
    "gfx_launch_counts": (C.c_int, [C.POINTER(_i64), C.c_int]),
}

STAGES = ("pack", "csr", "core_rows", "input", "aggregate", "mlp", "head",
          "fused_layer", "topk", "build", "align")

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

for _name, (_res, _args) in _SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here = ABI drift
    _fn.restype, _fn.argtypes = _res, _args

if lib.gfx_abi_version() != 1:
    raise NativeLibraryMissing("libgfx.so ABI version mismatch; rebuild it")


def check(status: int) -> None:
    if status != 0:
        message = lib.gfx_last_error().decode("utf-8", "replace")
        raise NativeError(f"libgfx error {status}: {message}")


def model_create(folded) -> int:
    """Upload FoldedWeights to the current CUDA device; returns a handle."""
    keep = {}

    def ptr(name):
        arr = np.ascontiguousarray(getattr(folded, name), dtype=np.float32)
        keep[name] = arr
        return arr.ctypes.data_as(_p)

    cfg = folded.cfg
    s = FoldedWeightsStruct(
        hidden=cfg.hidden, layers=cfg.layers, out_dim=cfg.out_dim,
        feature_dim=cfg.feature_dim, edge_dim=cfg.edge_dim,
        **{n: ptr(n) for n in ("w_in", "b_in", "table", "eps1", "w1", "b1",
                               "w2", "b2", "ln_g", "ln_b", "wa", "ba", "wb",
                               "bb")})
    handle = _p()
    check(lib.gfx_model_create(C.byref(s), C.byref(handle)))
    return handle.value


def model_destroy(handle) -> None:
    if handle:
        lib.gfx_model_destroy(_p(handle))


def launch_counts(reset: bool = False) -> dict:
    buf = (_i64 * len(STAGES))()
    check(lib.gfx_launch_counts(buf, 1 if reset else 0))
    return dict(zip(STAGES, list(buf)))


def profile_enable(*stages: str) -> None:
    mask = 0
    for name in stages:
        mask |= 1 << STAGES.index(name)
    check(lib.gfx_profile_enable(mask))


def profile_read(stage: str, reset: bool = True) -> tuple:
    """(total device milliseconds, number of timed calls) for one stage."""
    ms, calls = C.c_double(0), _i64(0)
    check(lib.gfx_profile_read(STAGES.index(stage), C.byref(ms), C.byref(calls),
                               1 if reset else 0))
    return ms.value, calls.value
