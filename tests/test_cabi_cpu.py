"""The C-ABI shared library loads and exports every symbol include/quanta_b200.h
declares (no compute calls — there is no GPU where this runs), and the host
layer fails loudly instead of falling back."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT
from quanta_b200 import _lib


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "quanta_b200.h")).read()
    return sorted(set(re.findall(r"QUANTA_API\s+[\w\s\*]+?\b(quanta_\w+)\s*\(", text)))


def test_header_declares_expected_entry_points():
    names = declared_symbols()
    for want in ["quanta_quantize_affine", "quanta_dequantize_affine", "quanta_pack4", "quanta_unpack4",
                 "quanta_backend_quantize", "quanta_backend_dequantize", "quanta_gemm_wna16",
                 "quanta_int8_outlier_matmul", "quanta_workspace_bytes", "quanta_error_string", "quanta_abi_version"]:
        assert want in names


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    h = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(h, name), f"{name} declared in include/quanta_b200.h but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature in quanta_b200/_lib.py"


def test_abi_version_and_error_strings():
    h = _lib.lib()
    assert h.quanta_abi_version() == 1
    assert h.quanta_error_string(0) == b"ok"
    assert b"invalid" in h.quanta_error_string(-1)
    assert b"workspace" in h.quanta_error_string(-3)
    assert h.quanta_workspace_bytes(_lib.OP_QUANTIZE_AFFINE, 4096, 4096) >= 256


def test_argument_errors_without_gpu():
    """Argument validation happens before any CUDA call."""
    h = _lib.lib()
    assert h.quanta_pack4(None, 4, None, None) == -1
    assert h.quanta_quantize_affine(None, 0, 1, 64, 2, 64, 4, 1, None, None, None, None, 0, None) == -1
    buf = ctypes.create_string_buffer(256)
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert h.quanta_quantize_affine(p, 0, 1, 100, 2, 64, 4, 1, p, p, p, None, 0, None) == -1     # 100 % 64
    assert h.quanta_quantize_affine(p, 0, 1, 64, 2, 64, 5, 0, p, p, p, None, 0, None) == -1      # bits
    assert h.quanta_quantize_affine(p, 0, 1, 64, 0, 0, 8, 0, p, p, p, p, 16, None) == -3         # workspace


def test_nf4_levels_need_no_gpu_and_match_the_oracle():
    """quanta_nf4_levels copies the library's one NF4 table on the host: no CUDA context, the oracle's bits."""
    import numpy as np
    from oracle import oracle_np as O
    buf = (ctypes.c_float * 16)()
    assert _lib.lib().quanta_nf4_levels(buf) == 0
    assert np.array_equal(np.frombuffer(buf, np.float32).view(np.uint32), O.NF4_LEVELS.view(np.uint32))
    assert _lib.lib().quanta_nf4_levels(None) == -1


def test_no_cpu_fallback():
    import quanta_b200 as Q
    from quanta_b200.backends.cuda import quantize_8bit_cuda
    x = torch.randn(8, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Q.quantize_8bit(x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        quantize_8bit_cuda(x, False, True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Q.pack_4bit_tensor(torch.zeros(4, dtype=torch.uint8))


def test_missing_extension_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libquanta_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.lib()


def test_error_behaviour_mirrors_reference():
    import quanta_b200 as Q
    x = torch.randn(4)
    with pytest.raises(ValueError, match="Unknown quantization type"):        # functional/quantization.py:18,31
        Q.quantize_8bit(x, quant_type="bogus")
    with pytest.raises(ValueError, match="Unknown quantization type"):
        Q.dequantize_4bit(x, x, x, quant_type="bogus")
    with pytest.raises(ValueError, match="Input tensor must be uint8"):        # utils/utils.py:25-26
        Q.pack_4bit_tensor(torch.zeros(4, dtype=torch.int32))


def test_workspace_sizes_are_small():
    """Per-tensor mode needs a fixed ~150 KB (partials of one CTA per SM for the single-launch kernels);
    dim-0 mode scales with the column count only."""
    h = _lib.lib()
    assert h.quanta_workspace_bytes(_lib.OP_QUANTIZE_AFFINE, 1, 1) < (1 << 18)
    assert h.quanta_workspace_bytes(_lib.OP_QUANTIZE_AFFINE, 11008, 4096) < (4 << 20)
    assert h.quanta_workspace_bytes(_lib.OP_BACKEND_DEQUANTIZE, 4096, 4096) == 256
