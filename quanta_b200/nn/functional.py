"""Host wrappers of the fused dequantize-then-matmul entry points."""
from __future__ import annotations

import torch

from .. import _host, _lib


def _check_weight_args(x, wq, params, N, K, bits, blocksize, what):
    """The kernels read ``wq`` as bytes and every parameter tensor as float32 through raw pointers: anything
    else (a buffer that ``module.half()`` cast to 16 bits, another device, a strided view, the wrong number
    of blocks) would be silently wrong and read out of bounds — refuse it here."""
    if blocksize <= 0 or K % blocksize:
        raise ValueError(f"{what}: in_features ({K}) must be a multiple of blocksize ({blocksize})")
    if not isinstance(wq, torch.Tensor) or wq.dtype != torch.uint8:
        raise TypeError(f"{what}: quantized weight must be a uint8 tensor")
    if wq.device != x.device or not wq.is_contiguous():
        raise ValueError(f"{what}: quantized weight must be contiguous and on {x.device}")
    if wq.numel() != N * K * bits // 8:
        raise ValueError(f"{what}: quantized weight holds {wq.numel()} bytes, expected {N * K * bits // 8} "
                         f"([{N}, {K}] at {bits} bits)")
    for name, t in params:
        if not isinstance(t, torch.Tensor) or t.dtype != torch.float32:
            raise TypeError(f"{what}: {name} must be a float32 tensor (got "
                            f"{getattr(t, 'dtype', type(t).__name__)}); quantization parameters are never cast with the module")
        if t.device != x.device or not t.is_contiguous():
            raise ValueError(f"{what}: {name} must be contiguous and on {x.device}")
        if t.numel() != N * K // blocksize:
            raise ValueError(f"{what}: {name} holds {t.numel()} values, expected {N * K // blocksize} "
                             f"(one per block of {blocksize})")


def linear_wna16(x, wq, scale, zp, bias=None, bits=4, blocksize=64, out_features=None, in_features=None):
    """y = x @ dequant(Wq).T + bias on the tcgen05 tensor cores.

    x      [..., K]   float16 / bfloat16 (CUDA)
    wq     bits=8: uint8 [N, K];  bits=4: nibble-packed uint8 [N*K/2] or [N, K/2]
           (``pack_4bit_tensor`` layout: even k -> low nibble)
    scale, zp  float32 [N*K/blocksize] — convention A, blockwise along K
           (``quantize_*bit(w, blocksize=B)``), blocksize = 64 * 2^j
    """
    _host.require_cuda(x, "x")
    if x.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError("x must be float16 or bfloat16")
    K = x.shape[-1]
    if in_features is not None and in_features != K:
        raise ValueError(f"x has {K} features, layer expects {in_features}")
    N = out_features if out_features is not None else (wq.shape[0] if wq.dim() == 2 else None)
    if N is None:
        raise ValueError("out_features is required for flat packed weights")
    if bits not in (4, 8):
        raise ValueError("bits must be 4 or 8")
    _check_weight_args(x, wq, (("scale", scale), ("zero_point", zp)), N, K, bits, blocksize, "linear_wna16")
    x2 = x.reshape(-1, K)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    M = x2.shape[0]
    dev = x.device
    y = torch.empty((M, N), dtype=x.dtype, device=dev)
    if M == 0:
        return y.reshape(*x.shape[:-1], N)
    if bias is not None and (bias.dtype != x.dtype or bias.device != dev or not bias.is_contiguous()):
        bias = bias.to(device=dev, dtype=x.dtype).contiguous()
    with _host.device_guard(dev):
        ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, N))
        st = _lib.lib().quanta_gemm_wna16(x2.data_ptr(), _host.dtype_code(x2), wq.data_ptr(), bits, scale.data_ptr(),
                                          zp.data_ptr(), blocksize, bias.data_ptr() if bias is not None else None,
                                          y.data_ptr(), M, N, K, ws.data_ptr(), ws.numel(), _host.stream_ptr(dev))
    _lib.check(st, "quanta_gemm_wna16")
    return y.reshape(*x.shape[:-1], N)


def linear_wna16_scatter(x, wq, scale, zp, bias, outs, col0, bits=4, blocksize=64, out_features=None, sync=None):
    """``linear_wna16`` whose epilogue writes this rank's output columns into every buffer
    of ``outs``: ``y_o[:, col0:col0+N] = x @ dequant(Wq).T + bias`` for each ``y_o``.

    outs   (device pointers, ldy): [M, ldy] buffers of x's dtype with the same row pitch —
           the local output and the peer-mapped outputs of the other ranks
    sync   optional (flag_ptrs, rank, world, epoch_counter_ptr): synchronise the ranks inside the kernel
           (``quanta_gemm_wna16_scatter_sync``; decode-sized batches only)
    Returns True when the ranks were synchronised in the kernel, else False: the caller
    then synchronises the ranks itself before reading."""
    import ctypes
    _host.require_cuda(x, "x")
    if x.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError("x must be float16 or bfloat16")
    K = x.shape[-1]
    N = out_features if out_features is not None else wq.shape[0]
    x2 = x.reshape(-1, K)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    M = x2.shape[0]
    ptrs, ldy = outs
    if M == 0 or N == 0:
        return False
    _check_weight_args(x, wq, (("scale", scale), ("zero_point", zp)), N, K, bits, blocksize, "linear_wna16_scatter")
    dev = x.device
    if bias is not None and (bias.dtype != x.dtype or bias.device != dev or not bias.is_contiguous()):
        bias = bias.to(device=dev, dtype=x.dtype).contiguous()
    arr = (ctypes.c_void_p * len(ptrs))(*ptrs)
    if sync is not None and M <= 16:
        flag_ptrs, rank, world, epoch_ptr = sync
        farr = (ctypes.c_void_p * len(flag_ptrs))(*flag_ptrs)
        with _host.device_guard(dev):
            ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, N))
            st = _lib.lib().quanta_gemm_wna16_scatter_sync(x2.data_ptr(), _host.dtype_code(x2), wq.data_ptr(), bits,
                                                           scale.data_ptr(), zp.data_ptr(), blocksize,
                                                           bias.data_ptr() if bias is not None else None, arr, len(ptrs), ldy,
                                                           col0, M, N, K, ws.data_ptr(), ws.numel(), farr, rank, world,
                                                           epoch_ptr, _host.stream_ptr(dev))
        if st == 0:
            return True
        if st != _lib.E_UNSUPPORTED:
            _lib.check(st, "quanta_gemm_wna16_scatter_sync")
    with _host.device_guard(dev):
        ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, N))
        st = _lib.lib().quanta_gemm_wna16_scatter(x2.data_ptr(), _host.dtype_code(x2), wq.data_ptr(), bits,
                                                  scale.data_ptr(), zp.data_ptr(), blocksize,
                                                  bias.data_ptr() if bias is not None else None, arr, len(ptrs), ldy,
                                                  col0, M, N, K, ws.data_ptr(), ws.numel(), _host.stream_ptr(dev))
    _lib.check(st, "quanta_gemm_wna16_scatter")
    return False


def linear_nf4a16(x, wq, absmax, bias=None, blocksize=64, out_features=None, in_features=None):
    """y = x @ (nf4_level[Wq] * absmax).T + bias on the tcgen05 tensor cores — the forward of
    ``Linear4bit(quant_type="nf4")`` (the reference's default, Quanta/nn/linear.py:58).

    wq      nibble-packed NF4 codes, uint8 [N*K/2] or [N, K/2] (``quantize_4bit(w, "nf4", blocksize=B, packed=True)``)
    absmax  float32 [N*K/blocksize], blocksize = 64 * 2^j dividing K"""
    _host.require_cuda(x, "x")
    if x.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError("x must be float16 or bfloat16")
    K = x.shape[-1]
    if in_features is not None and in_features != K:
        raise ValueError(f"x has {K} features, layer expects {in_features}")
    N = out_features if out_features is not None else (wq.shape[0] if wq.dim() == 2 else None)
    if N is None:
        raise ValueError("out_features is required for flat packed weights")
    _check_weight_args(x, wq, (("absmax", absmax),), N, K, 4, blocksize, "linear_nf4a16")
    x2 = x.reshape(-1, K)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    M = x2.shape[0]
    dev = x.device
    y = torch.empty((M, N), dtype=x.dtype, device=dev)
    if M == 0:
        return y.reshape(*x.shape[:-1], N)
    if bias is not None and (bias.dtype != x.dtype or bias.device != dev or not bias.is_contiguous()):
        bias = bias.to(device=dev, dtype=x.dtype).contiguous()
    with _host.device_guard(dev):
        ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, N))
        st = _lib.lib().quanta_gemm_nf4a16(x2.data_ptr(), _host.dtype_code(x2), wq.data_ptr(), absmax.data_ptr(),
                                           blocksize, bias.data_ptr() if bias is not None else None, y.data_ptr(),
                                           M, N, K, ws.data_ptr(), ws.numel(), _host.stream_ptr(dev))
    _lib.check(st, "quanta_gemm_nf4a16")
    return y.reshape(*x.shape[:-1], N)


def _dgrad_args(dy, wq, bits, out_features, in_features, what):
    """dy as the [M, round_up(N, 8)] matrix the dgrad entries read (zero columns past N), and (N, K)."""
    _host.require_cuda(dy, "dy")
    if dy.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError("dy must be float16 or bfloat16")
    N = dy.shape[-1]
    if out_features is not None and out_features != N:
        raise ValueError(f"{what}: dy has {N} features, layer has {out_features} outputs")
    if in_features is None:
        if N == 0 or not isinstance(wq, torch.Tensor):
            raise ValueError(f"{what}: in_features is required")
        in_features = wq.numel() * 8 // bits // N
    dy2 = dy.reshape(-1, N)
    if N % 8:
        dy2 = torch.nn.functional.pad(dy2, (0, 8 - N % 8))
    if not dy2.is_contiguous():
        dy2 = dy2.contiguous()
    return dy2, N, in_features


def linear_wna16_dgrad(dy, wq, scale, zp, bits=4, blocksize=64, out_features=None, in_features=None):
    """dx = dy @ dequant(Wq): the input gradient of ``linear_wna16`` for a frozen weight, with the weights
    dequantized to bit-for-bit the 16-bit values the forward multiplies with.

    dy     [..., N]   float16 / bfloat16 (CUDA);  returns dx [..., K] in dy's dtype
    wq, scale, zp, bits, blocksize as for ``linear_wna16``"""
    if bits not in (4, 8):
        raise ValueError("bits must be 4 or 8")
    dy2, N, K = _dgrad_args(dy, wq, bits, out_features, in_features, "linear_wna16_dgrad")
    _check_weight_args(dy, wq, (("scale", scale), ("zero_point", zp)), N, K, bits, blocksize, "linear_wna16_dgrad")
    M = dy2.shape[0]
    dev = dy.device
    dx = torch.empty((M, K), dtype=dy.dtype, device=dev)
    if M == 0 or N == 0:
        return dx.zero_().reshape(*dy.shape[:-1], K)
    with _host.device_guard(dev):
        ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, K))
        st = _lib.lib().quanta_gemm_wna16_dgrad(dy2.data_ptr(), _host.dtype_code(dy2), wq.data_ptr(), bits, scale.data_ptr(),
                                                zp.data_ptr(), blocksize, dx.data_ptr(), M, N, K, ws.data_ptr(), ws.numel(),
                                                _host.stream_ptr(dev))
    _lib.check(st, "quanta_gemm_wna16_dgrad")
    return dx.reshape(*dy.shape[:-1], K)


def linear_nf4a16_dgrad(dy, wq, absmax, blocksize=64, out_features=None, in_features=None):
    """dx = dy @ (nf4_level[Wq] * absmax): the input gradient of ``linear_nf4a16`` for a frozen weight."""
    dy2, N, K = _dgrad_args(dy, wq, 4, out_features, in_features, "linear_nf4a16_dgrad")
    _check_weight_args(dy, wq, (("absmax", absmax),), N, K, 4, blocksize, "linear_nf4a16_dgrad")
    M = dy2.shape[0]
    dev = dy.device
    dx = torch.empty((M, K), dtype=dy.dtype, device=dev)
    if M == 0 or N == 0:
        return dx.zero_().reshape(*dy.shape[:-1], K)
    with _host.device_guard(dev):
        ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, K))
        st = _lib.lib().quanta_gemm_nf4a16_dgrad(dy2.data_ptr(), _host.dtype_code(dy2), wq.data_ptr(), absmax.data_ptr(),
                                                 blocksize, dx.data_ptr(), M, N, K, ws.data_ptr(), ws.numel(),
                                                 _host.stream_ptr(dev))
    _lib.check(st, "quanta_gemm_nf4a16_dgrad")
    return dx.reshape(*dy.shape[:-1], K)


class LinearWNA16Function(torch.autograd.Function):
    """``linear_wna16`` with a backward for x and bias; the quantized weight is frozen and gets no gradient.

    ``bias`` is the parameter the gradient goes to; ``bias_k`` is the same values as the kernel reads them
    (x's dtype, contiguous).  A double backward is not supported."""

    @staticmethod
    def forward(ctx, x, bias, bias_k, wq, scale, zp, bits, blocksize, out_features, in_features):
        ctx.save_for_backward(wq, scale, zp)
        ctx.meta = (bits, blocksize, out_features, in_features)
        ctx.bias_dtype = bias.dtype if bias is not None else None
        return linear_wna16(x, wq, scale, zp, bias_k, bits=bits, blocksize=blocksize, out_features=out_features,
                            in_features=in_features)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        wq, scale, zp = ctx.saved_tensors
        bits, blocksize, N, K = ctx.meta
        dx = db = None
        if ctx.needs_input_grad[0]:
            dx = linear_wna16_dgrad(dy, wq, scale, zp, bits=bits, blocksize=blocksize, out_features=N, in_features=K)
        if ctx.needs_input_grad[1]:
            db = dy.reshape(-1, N).sum(0, dtype=torch.float32).to(ctx.bias_dtype)
        return dx, db, None, None, None, None, None, None, None, None


class LinearNF4A16Function(torch.autograd.Function):
    """``linear_nf4a16`` with a backward for x and bias (see ``LinearWNA16Function``)."""

    @staticmethod
    def forward(ctx, x, bias, bias_k, wq, absmax, blocksize, out_features, in_features):
        ctx.save_for_backward(wq, absmax)
        ctx.meta = (blocksize, out_features, in_features)
        ctx.bias_dtype = bias.dtype if bias is not None else None
        return linear_nf4a16(x, wq, absmax, bias_k, blocksize=blocksize, out_features=out_features, in_features=in_features)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        wq, absmax = ctx.saved_tensors
        blocksize, N, K = ctx.meta
        dx = db = None
        if ctx.needs_input_grad[0]:
            dx = linear_nf4a16_dgrad(dy, wq, absmax, blocksize=blocksize, out_features=N, in_features=K)
        if ctx.needs_input_grad[1]:
            db = dy.reshape(-1, N).sum(0, dtype=torch.float32).to(ctx.bias_dtype)
        return dx, db, None, None, None, None, None, None


def rowwise_quantize_sym(weight):
    """Static int8 weight codes for the outlier-split matmul: convention-B
    symmetric 8-bit with one multiplier per OUTPUT row, i.e.
    ``quantize_8bit_cuda(w.t(), per_channel=True, symmetric=True)``
    (Quanta/backends/cpu/quantization.py:29-50) transposed back and re-centred.
    Returns (qw int8 [N, K] = code - 128, cw float32 [N] = 127 / absmax)."""
    from ..backends.cuda.quantization import quantize_8bit_cuda
    _host.require_cuda(weight, "weight")
    q, scale, _ = quantize_8bit_cuda(weight.detach().float().t().contiguous(), True, True)
    qw = (q.t().to(torch.int16) - 128).to(torch.int8).contiguous()
    return qw, scale.reshape(-1).contiguous()


def int8_outlier_matmul(x, qw, cw, threshold=6.0, bias=None):
    """LLM.int8()-style y = x @ W.T + bias over int8 weight codes (row G3):
    feature columns of ``x`` whose absolute maximum exceeds ``threshold`` go
    through a 16-bit product with the dequantized weight columns, the rest
    through int8 x int8 -> int32 on the tensor cores with row-wise absmax
    scales for ``x`` (semantics: oracle/oracle_np.py:int8_outlier_matmul).

    x [..., K] float16 / bfloat16; qw int8 [N, K]; cw float32 [N]."""
    _host.require_cuda(x, "x")
    if x.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError("x must be float16 or bfloat16")
    N, K = _check_rowwise_args(x, qw, cw)
    if x.shape[-1] != K:
        raise ValueError(f"x has {x.shape[-1]} features, weight expects {K}")
    x2 = x.reshape(-1, K)
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    M = x2.shape[0]
    dev = x.device
    y = torch.empty((M, N), dtype=x.dtype, device=dev)
    if M == 0:
        return y.reshape(*x.shape[:-1], N)
    if bias is not None and (bias.dtype != x.dtype or bias.device != dev or not bias.is_contiguous()):
        bias = bias.to(device=dev, dtype=x.dtype).contiguous()
    with _host.device_guard(dev):
        ws = _host.workspace(dev, _host.workspace_bytes(_lib.OP_INT8_OUTLIER, M, K))
        st = _lib.lib().quanta_int8_outlier_matmul(x2.data_ptr(), _host.dtype_code(x2), qw.data_ptr(), cw.data_ptr(),
                                                   float(threshold), bias.data_ptr() if bias is not None else None,
                                                   y.data_ptr(), M, N, K, ws.data_ptr(), ws.numel(),
                                                   _host.stream_ptr(dev))
    _lib.check(st, "quanta_int8_outlier_matmul")
    return y.reshape(*x.shape[:-1], N)


def _check_rowwise_args(x, qw, cw):
    """qw int8 [N, K] and cw float32 [N] as the int8 kernels read them; returns (N, K)."""
    if not isinstance(qw, torch.Tensor) or qw.dtype != torch.int8 or qw.dim() != 2:
        raise TypeError("qw must be an int8 [N, K] tensor")
    N, K = qw.shape
    if qw.device != x.device or not qw.is_contiguous():
        raise ValueError(f"qw must be contiguous and on {x.device}")
    if not isinstance(cw, torch.Tensor) or cw.dtype != torch.float32 or cw.numel() != N or cw.device != x.device or not cw.is_contiguous():
        raise TypeError(f"cw must be a contiguous float32 tensor of {N} row multipliers on {x.device}")
    return N, K


def int8_outlier_dgrad(dy, qw, cw):
    """dx = dy @ W16 with ``W16[n, k] = round_act(qw[n, k] / cw[n])`` (an IEEE divide, then one rounding to
    dy's dtype): the input gradient of ``int8_outlier_matmul`` for a frozen weight.  W16 is bit for bit the
    weight the forward multiplies its outlier columns with, and ``Linear8bitLt.dequantize_weight(dtype)``.
    The gradient is straight-through: the int8 quantization of x and the outlier set do not enter, so the
    threshold is not an argument.

    dy [..., N] float16 / bfloat16 (CUDA); qw int8 [N, K] with K % 16 == 0; cw float32 [N].
    Returns dx [..., K] in dy's dtype (fp32 accumulation)."""
    _host.require_cuda(dy, "dy")
    if dy.dtype not in (torch.float16, torch.bfloat16):
        raise TypeError("dy must be float16 or bfloat16")
    N, K = _check_rowwise_args(dy, qw, cw)
    if dy.shape[-1] != N:
        raise ValueError(f"int8_outlier_dgrad: dy has {dy.shape[-1]} features, weight has {N} outputs")
    if dy.numel() == 0:
        return torch.zeros((*dy.shape[:-1], K), dtype=dy.dtype, device=dy.device)
    dy2, N, K = _dgrad_args(dy, qw, 8, N, K, "int8_outlier_dgrad")
    M = dy2.shape[0]
    dev = dy.device
    dx = torch.empty((M, K), dtype=dy.dtype, device=dev)
    with _host.device_guard(dev):
        ws = _host.gemm_workspace(dev, _host.workspace_bytes(_lib.OP_GEMM, M, K))
        st = _lib.lib().quanta_int8_outlier_dgrad(dy2.data_ptr(), _host.dtype_code(dy2), qw.data_ptr(), cw.data_ptr(),
                                                  dx.data_ptr(), M, N, K, ws.data_ptr(), ws.numel(), _host.stream_ptr(dev))
    _lib.check(st, "quanta_int8_outlier_dgrad")
    return dx.reshape(*dy.shape[:-1], K)


class Int8OutlierMatmulFunction(torch.autograd.Function):
    """``int8_outlier_matmul`` with the straight-through backward for x and bias (bitsandbytes'
    ``MatMul8bitLt``): ``dx = dy @ W16`` through ``int8_outlier_dgrad``, ``db = dy.sum(0)`` accumulated in fp32.
    Only qw and cw are saved.  ``bias`` / ``bias_k`` as in ``LinearWNA16Function``; no double backward."""

    @staticmethod
    def forward(ctx, x, bias, bias_k, qw, cw, threshold):
        ctx.save_for_backward(qw, cw)
        ctx.bias_dtype = bias.dtype if bias is not None else None
        return int8_outlier_matmul(x, qw, cw, threshold, bias_k)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        qw, cw = ctx.saved_tensors
        dx = db = None
        if ctx.needs_input_grad[0]:
            dx = int8_outlier_dgrad(dy, qw, cw)
        if ctx.needs_input_grad[1]:
            db = dy.reshape(-1, qw.shape[0]).sum(0, dtype=torch.float32).to(ctx.bias_dtype)
        return dx, db, None, None, None, None

