"""The input-gradient entries of the dequant-GEMM reject bad arguments before any CUDA call
(no GPU here: a call that got as far as the device would not return these codes)."""
import ctypes

from quanta_b200 import _lib

BF16 = _lib.BF16


def _bufs():
    buf = ctypes.create_string_buffer(1 << 16)
    addr = (ctypes.addressof(buf) + 255) // 256 * 256        # 16-byte aligned operands
    return buf, ctypes.c_void_p(addr)


def test_wna16_dgrad_rejects_bad_arguments():
    h = _lib.lib()
    _keep, p = _bufs()
    ws = h.quanta_workspace_bytes(_lib.OP_GEMM, 16, 128)
    f = h.quanta_gemm_wna16_dgrad
    # dy, act, wq, bits, scale, zp, block, dx, M, N, K, ws, ws_bytes, stream
    assert f(None, BF16, p, 4, p, p, 64, p, 16, 64, 128, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, None, 4, p, p, 64, p, 16, 64, 128, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, 4, None, p, 64, p, 16, 64, 128, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, 4, p, None, 64, p, 16, 64, 128, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, 4, p, p, 64, None, 16, 64, 128, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, 5, p, p, 64, p, 16, 64, 128, p, ws, None) == _lib.E_INVAL        # bits
    assert f(p, BF16, p, 8, p, p, 128, p, 16, 64, 192, p, ws, None) == _lib.E_INVAL       # K % block
    assert f(p, BF16, p, 4, p, p, 96, p, 16, 64, 192, p, ws, None) == _lib.E_INVAL        # block % 64
    assert f(p, BF16, p, 4, p, p, 192, p, 16, 64, 192, p, ws, None) == _lib.E_UNSUPPORTED  # block != 64 * 2^j
    assert f(p, BF16, p, 4, p, p, 64, p, 0, 64, 128, p, ws, None) == _lib.E_INVAL         # M
    assert f(p, BF16, p, 4, p, p, 64, p, 16, 64, 128, p, 16, None) == _lib.E_WORKSPACE    # workspace too small
    assert f(p, BF16, p, 4, p, p, 64, p, 16, 64, 128, None, ws, None) == _lib.E_WORKSPACE


def test_nf4a16_dgrad_rejects_bad_arguments():
    h = _lib.lib()
    _keep, p = _bufs()
    ws = h.quanta_workspace_bytes(_lib.OP_GEMM, 300, 256)
    f = h.quanta_gemm_nf4a16_dgrad
    # dy, act, wq, absmax, block, dx, M, N, K, ws, ws_bytes, stream
    assert f(None, BF16, p, p, 64, p, 300, 1001, 256, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, None, p, 64, p, 300, 1001, 256, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, None, 64, p, 300, 1001, 256, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, p, 64, None, 300, 1001, 256, p, ws, None) == _lib.E_INVAL
    assert f(p, BF16, p, p, 128, p, 300, 1001, 320, p, ws, None) == _lib.E_INVAL        # K % block
    assert f(p, BF16, p, p, 64, p, 300, 1001, 256, p, 1024, None) == _lib.E_WORKSPACE
    assert f(p, 7, p, p, 64, p, 300, 1001, 256, p, ws, None) == _lib.E_INVAL          # act_dtype

