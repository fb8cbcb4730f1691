"""ctypes loader for libquanta_b200.so — the C-ABI declared in include/quanta_b200.h.

There is deliberately NO fallback: if the shared library is missing or a call
returns a non-zero status the caller gets an exception (north_star: "no CPU
fallback"; unlike Quanta/backends/__init__.py:25-26, which swallows the
ImportError and silently stays on the CPU path).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libquanta_b200.so")

MODE_TENSOR, MODE_DIM0, MODE_BLOCK = 0, 1, 2
E_INVAL, E_UNSUPPORTED, E_WORKSPACE, E_DRIVER = -1, -2, -3, -4        # include/quanta_b200.h
F32, F16, BF16 = 0, 1, 2
OP_QUANTIZE_AFFINE, OP_BACKEND_QUANTIZE, OP_BACKEND_DEQUANTIZE, OP_GEMM, OP_INT8_OUTLIER, OP_BASE_QUANTIZE = range(6)

# every symbol include/quanta_b200.h declares: name -> (restype, argtypes)
_i64, _int, _vp, _sz, _f = C.c_int64, C.c_int, C.c_void_p, C.c_size_t, C.c_float
SIGNATURES = {
    "quanta_abi_version": (_int, []),
    "quanta_error_string": (C.c_char_p, [_int]),
    "quanta_workspace_bytes": (_sz, [_int, _i64, _i64]),
    "quanta_quantize_affine": (_int, [_vp, _int, _i64, _i64, _int, _i64, _int, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "quanta_quantize_block_batch": (_int, [_vp, _vp, _int, _int, _i64, _int, _int, _vp, _vp, _vp, _vp]),
    "quanta_dequantize_affine": (_int, [_vp, _int, _i64, _i64, _int, _i64, _vp, _vp, _vp, _int, _vp]),
    "quanta_dequantize_block_batch": (_int, [_vp, _vp, _int, _int, _i64, _vp, _vp, _vp, _int, _vp]),
    "quanta_nf4_levels": (_int, [_vp]),
    "quanta_quantize_nf4": (_int, [_vp, _int, _i64, _i64, _int, _vp, _vp, _vp]),
    "quanta_dequantize_nf4": (_int, [_vp, _int, _i64, _i64, _vp, _vp, _int, _vp]),
    "quanta_pack4": (_int, [_vp, _i64, _vp, _vp]),
    "quanta_unpack4": (_int, [_vp, _i64, _vp, _vp]),
    "quanta_pack4_hi": (_int, [_vp, _i64, _vp, _vp]),
    "quanta_unpack4_hi": (_int, [_vp, _i64, _vp, _vp]),
    "quanta_backend_quantize": (_int, [_vp, _int, _i64, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "quanta_backend_dequantize": (_int, [_vp, _i64, _i64, _i64, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "quanta_base_quantize": (_int, [_vp, _int, _i64, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "quanta_base_dequantize": (_int, [_vp, _i64, _i64, _i64, _int, _int, _vp, _vp, _vp, _vp]),
    "quanta_convert_linear": (_int, [_vp, _i64, _vp, _vp, _int, _vp, _vp, _vp, _vp, _sz, _vp]),
    "quanta_nf8_levels": (_int, [_vp]),
    "quanta_quantize_nf8": (_int, [_vp, _int, _i64, _i64, _vp, _vp, _vp]),
    "quanta_dequantize_nf8": (_int, [_vp, _i64, _i64, _vp, _vp, _int, _vp]),
    "quanta_quantize_fp": (_int, [_vp, _int, _i64, _int, _vp, _vp]),
    "quanta_dequantize_fp": (_int, [_vp, _i64, _int, _int, _vp, _int, _vp]),
    "quanta_gemm_wna16": (_int, [_vp, _int, _vp, _int, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _i64, _vp, _sz, _vp]),
    "quanta_gemm_wna16_scatter": (_int, [_vp, _int, _vp, _int, _vp, _vp, _i64, _vp, _vp, _int, _i64, _i64, _i64, _i64, _i64, _vp,
                                         _sz, _vp]),
    "quanta_gemm_wna16_scatter_sync": (_int, [_vp, _int, _vp, _int, _vp, _vp, _i64, _vp, _vp, _int, _i64, _i64, _i64, _i64, _i64, _vp,
                                              _sz, _vp, _int, _int, _vp, _vp]),
    "quanta_peer_barrier": (_int, [_vp, _int, _int, _vp, _vp]),
    "quanta_gemm_nf4a16": (_int, [_vp, _int, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _i64, _vp, _sz, _vp]),
    "quanta_gemm_wna16_dgrad": (_int, [_vp, _int, _vp, _int, _vp, _vp, _i64, _vp, _i64, _i64, _i64, _vp, _sz, _vp]),
    "quanta_gemm_nf4a16_dgrad": (_int, [_vp, _int, _vp, _vp, _i64, _vp, _i64, _i64, _i64, _vp, _sz, _vp]),
    "quanta_int8_outlier_matmul": (_int, [_vp, _int, _vp, _vp, _f, _vp, _vp, _i64, _i64, _i64, _vp, _sz, _vp]),
    "quanta_int8_outlier_dgrad": (_int, [_vp, _int, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _sz, _vp]),
}

_lib = None


class QuantaError(RuntimeError):
    """A C-ABI call returned a non-zero status."""


def build(verbose=False):
    """Compile libquanta_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", os.path.join(_PKG, "csrc"), "-j8"], capture_output=True, text=True)
    if verbose or out.returncode:
        print(out.stdout[-4000:], out.stderr[-4000:])
    if out.returncode:
        raise RuntimeError("building libquanta_b200.so failed")
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension is the only implementation of this path "
                "(no CPU fallback). Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C quanta_b200/csrc`.")
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype, fn.argtypes = res, args
        if h.quanta_abi_version() != 1:
            raise RuntimeError("libquanta_b200.so ABI version mismatch")
        _lib = h
    return _lib


def check(status, what):
    if status != 0:
        msg = lib().quanta_error_string(status).decode()
        raise QuantaError(f"{what} failed with status {status}: {msg}")
