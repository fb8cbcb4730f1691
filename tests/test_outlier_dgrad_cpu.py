"""The input-gradient entry of the outlier-split matmul rejects bad arguments before any CUDA call
(no GPU here: a call that got as far as the device would not return these codes)."""
import ctypes

from quanta_b200 import _lib

BF16 = _lib.BF16


def _bufs():
    buf = ctypes.create_string_buffer(1 << 16)
    addr = (ctypes.addressof(buf) + 255) // 256 * 256        # 16-byte aligned operands
    return buf, addr


def test_int8_outlier_dgrad_rejects_bad_arguments():
    h = _lib.lib()
    _keep, a = _bufs()
    p = ctypes.c_void_p(a)
    ws = h.quanta_workspace_bytes(_lib.OP_GEMM, 300, 336)
    f = h.quanta_int8_outlier_dgrad
    # dy, act, qw, cw, dx, M, N, K, ws, ws_bytes, stream
    assert f(None, BF16, p, p, p, 300, 1001, 336, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, None, p, p, 300, 1001, 336, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, None, p, 300, 1001, 336, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, p, None, 300, 1001, 336, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, p, p, 0, 1001, 336, p, ws, None) == _lib.E_INVAL           # M
    assert f(p, BF16, p, p, p, 300, 0, 336, p, ws, None) == _lib.E_INVAL            # N
    assert f(p, BF16, p, p, p, 300, 1001, 0, p, ws, None) == _lib.E_INVAL           # K
    assert f(p, BF16, p, p, p, 300, 1001, -16, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, p, p, 300, 1001, 328, p, ws, None) == _lib.E_UNSUPPORTED   # K % 16
    assert f(p, BF16, p, p, p, 300, 1001, 1 << 31, p, ws, None) == _lib.E_UNSUPPORTED
    assert f(ctypes.c_void_p(a + 8), BF16, p, p, p, 300, 1001, 336, p, ws, None) == _lib.E_UNSUPPORTED  # dy alignment
    assert f(p, BF16, ctypes.c_void_p(a + 8), p, p, 300, 1001, 336, p, ws, None) == _lib.E_UNSUPPORTED  # qw alignment
    assert f(p, 7, p, p, p, 300, 1001, 336, p, ws, None) == _lib.E_INVAL            # act_dtype
    assert f(p, BF16, p, p, p, 300, 1001, 336, p, 1024, None) == _lib.E_WORKSPACE   # workspace too small
    assert f(p, BF16, p, p, p, 300, 1001, 336, None, ws, None) == _lib.E_WORKSPACE
    assert f(p, BF16, p, p, p, 16, 64, 16, p, 16, None) == _lib.E_WORKSPACE

