"""Drop-in CUDA implementation of ``Quanta.functional.quantization`` ("linear").

Same names, argument meaning, return layout and error behaviour as the
reference (Quanta/functional/quantization.py:7-71), computed by the sm_100a
kernels behind include/quanta_b200.h:

    q_tensor, scale, zero_point = quantize_8bit(tensor)              # :20
    q_tensor, scale, zero_point = quantize_4bit(tensor, per_channel=True)
    x = dequantize_8bit(q_tensor, scale, zero_point)                 # :33

New keyword arguments default to the reference behaviour:
  blocksize=B  blockwise quantization — the reference's ``per_channel=True``
               branch applied to ``tensor.reshape(-1, B).t()`` (SURVEY Appendix
               A.1); ``scale`` / ``zero_point`` come back with shape [numel/B],
               codes keep the input's shape and order.
  packed=True  (4-bit) codes are returned nibble-packed as
               ``pack_4bit_tensor`` would (flat uint8 of ceil(numel/2)).
"""
from __future__ import annotations

import torch

from .. import _host, _lib

_levels = {}          # (quant_type, str(device)) -> the codebook's levels as a float32 tensor on that device


def _quantize_linear(tensor, bits, per_channel, blocksize, packed):
    _host.require_cuda(tensor)
    x = tensor.detach()
    if not x.is_contiguous():
        x = x.contiguous()
    code = _host.dtype_code(x)
    n = x.numel()
    if n == 0:
        raise RuntimeError("min(): cannot quantize an empty tensor")          # torch.min raises on empty input
    dev = x.device
    if blocksize is not None:
        B = int(blocksize)
        if B <= 0 or n % B:
            raise ValueError(f"numel ({n}) must be a multiple of blocksize ({blocksize})")
        mode, rows, cols, nparam, pshape = _lib.MODE_BLOCK, 1, n, n // B, (n // B,)
    elif per_channel:
        if x.dim() < 2:
            # the reference calls tensor.min(dim=None, keepdim=True) here, which raises
            raise ValueError("per_channel=True needs a tensor with dim() > 1")
        rows, cols = _host.rows_cols(x)
        mode, nparam, pshape, B = _lib.MODE_DIM0, cols, (1,) + tuple(x.shape[1:]), 0
    else:
        mode, rows, cols, nparam, pshape, B = _lib.MODE_TENSOR, 1, n, 1, (), 0
    with _host.device_guard(dev):
        scale = torch.empty(nparam, dtype=torch.float32, device=dev)
        zp = torch.empty(nparam, dtype=torch.float32, device=dev)
        q = torch.empty((n + 1) // 2 if packed else n, dtype=torch.uint8, device=dev)
        # only the two-pass modes need scratch: per-tensor partials, or per-column partials for dim 0
        ws_bytes = _host.workspace_bytes(_lib.OP_QUANTIZE_AFFINE, rows if mode == _lib.MODE_DIM0 else 1,
                                                     cols if mode == _lib.MODE_DIM0 else 1)
        ws = _host.quantize_workspace(dev, ws_bytes)
        st = _lib.lib().quanta_quantize_affine(x.data_ptr(), code, rows, cols, mode, B, bits, int(bool(packed)),
                                               q.data_ptr(), scale.data_ptr(), zp.data_ptr(),
                                               ws.data_ptr(), ws.numel(), _host.stream_ptr(dev))
        if st == -2 and packed:
            # odd block sizes: quantize unpacked, then pack (same bytes)
            q = torch.empty(n, dtype=torch.uint8, device=dev)
            st = _lib.lib().quanta_quantize_affine(x.data_ptr(), code, rows, cols, mode, B, bits, 0,
                                                   q.data_ptr(), scale.data_ptr(), zp.data_ptr(),
                                                   ws.data_ptr(), ws.numel(), _host.stream_ptr(dev))
            _lib.check(st, "quanta_quantize_affine")
            from ..utils.utils import pack_4bit_tensor
            q = pack_4bit_tensor(q)[0]
        else:
            _lib.check(st, "quanta_quantize_affine")
    if not packed:
        q = q.reshape(tensor.shape)
    return q, scale.reshape(pshape), zp.reshape(pshape)


def _codebook_levels(quant_type, device):
    import ctypes as C
    key = (quant_type, str(device))
    if key not in _levels:
        count, entry = (16, "quanta_nf4_levels") if quant_type == "nf4" else (256, "quanta_nf8_levels")
        buf = (C.c_float * count)()
        _lib.check(getattr(_lib.lib(), entry)(buf), entry)
        _levels[key] = torch.tensor(list(buf), dtype=torch.float32, device=device)
    return _levels[key]


def nf4_levels(device):
    """The 16 NF4 levels as a float32 tensor on ``device`` (second return value of the reference's
    ``quantize_4bit(..., quant_type="nf4")``, Quanta/functional/quantization.py:105-110)."""
    return _codebook_levels("nf4", device)


def nf8_levels(device):
    """The 256 nf8 levels ``tanh(2 * linspace(-1, 1, 256))`` exactly as the reference's torch computes them
    (second return value of ``quantize_8bit(..., quant_type="nf8")``, Quanta/functional/quantization.py:174-175)."""
    return _codebook_levels("nf8", device)


def _prep_input(tensor):
    _host.require_cuda(tensor)
    x = tensor.detach()
    if not x.is_contiguous():
        x = x.contiguous()
    return x, _host.dtype_code(x), x.numel(), x.device


def _prep_codes(q_tensor):
    """The codes argument of a dequantize call as a contiguous uint8 CUDA tensor."""
    _host.require_cuda(q_tensor, "q_tensor")
    q = q_tensor.detach()
    if q.dtype != torch.uint8:
        q = q.to(torch.uint8)
    if not q.is_contiguous():
        q = q.contiguous()
    return q


def _out_shape(q, packed, shape):
    """Shape of the dequantized output: the codes' shape, or for nibble-packed codes ``shape`` (default: two values per
    byte), which must need exactly the bytes ``q`` holds."""
    if not packed:
        return q.shape
    out_shape = torch.Size(shape) if shape is not None else torch.Size([q.numel() * 2])
    n = out_shape.numel()
    if q.numel() != (n + 1) // 2:
        # a wrong ``shape`` would make the kernel read past the packed buffer
        raise ValueError(f"packed codes hold {q.numel()} bytes, shape {tuple(out_shape)} needs {(n + 1) // 2}")
    return out_shape


def _check_nf4_blocksize(B, blocksize):
    if B and (B < 16 or B > 512 or (B & (B - 1))):
        raise ValueError(f"NF4 blocksize must be 16 * 2^j <= 512 (got {blocksize}); the affine formats take any block size")


def _quantize_codebook(tensor, quant_type, blocksize, packed=False):
    """NF4 / nf8: returns ``(codes, levels, abs_max)`` like the reference (:118, :183).  Only NF4 packs; nf8 leaves
    an unsupported block size to the C entry."""
    x, code, n, dev = _prep_input(tensor)
    if n == 0:
        raise RuntimeError("max(): cannot quantize an empty tensor")
    B = 0 if blocksize is None else int(blocksize)
    if B and n % B:
        raise ValueError(f"numel ({n}) must be a multiple of blocksize ({blocksize})")
    if quant_type == "nf4":
        _check_nf4_blocksize(B, blocksize)
    with _host.device_guard(dev):
        q = torch.empty((n + 1) // 2 if packed else n, dtype=torch.uint8, device=dev)
        absmax = torch.empty(n // B if B else 1, dtype=torch.float32, device=dev)
        if quant_type == "nf4":
            st = _lib.lib().quanta_quantize_nf4(x.data_ptr(), code, n, B, int(bool(packed)), q.data_ptr(),
                                                absmax.data_ptr(), _host.stream_ptr(dev))
        else:
            st = _lib.lib().quanta_quantize_nf8(x.data_ptr(), code, n, B, q.data_ptr(), absmax.data_ptr(),
                                                _host.stream_ptr(dev))
    _lib.check(st, f"quanta_quantize_{quant_type}")
    if not packed:
        q = q.reshape(tensor.shape)
    return q, _codebook_levels(quant_type, dev), (absmax if B else absmax.reshape(()))


def _dequantize_codebook(q_tensor, absmax, quant_type, blocksize, packed, shape, out_dtype):
    """``levels[q] * abs_max`` for NF4 (optionally nibble-packed) and nf8."""
    q = _prep_codes(q_tensor)
    dev = q.device
    absmax = torch.as_tensor(absmax, dtype=torch.float32, device=dev).reshape(-1).contiguous()
    out_shape = _out_shape(q, packed, shape)
    n = out_shape.numel()
    out = torch.empty(out_shape, dtype=out_dtype, device=dev)
    if n == 0:
        return out
    B = 0 if blocksize is None else int(blocksize)
    if quant_type == "nf4":
        _check_nf4_blocksize(B, blocksize)
    if (B and absmax.numel() != n // B) or (not B and absmax.numel() != 1):
        raise ValueError("absmax does not match blocksize")
    with _host.device_guard(dev):
        if quant_type == "nf4":
            st = _lib.lib().quanta_dequantize_nf4(q.data_ptr(), int(bool(packed)), n, B, absmax.data_ptr(),
                                                  out.data_ptr(), _host._DTYPE[out_dtype], _host.stream_ptr(dev))
        else:
            st = _lib.lib().quanta_dequantize_nf8(q.data_ptr(), n, B, absmax.data_ptr(), out.data_ptr(),
                                                  _host._DTYPE[out_dtype], _host.stream_ptr(dev))
    _lib.check(st, f"quanta_dequantize_{quant_type}")
    return out


def _quantize_fp(tensor, bits):
    """fp4 / fp8: returns ``(codes, None, exp_bias)`` like the reference (:144, :168)."""
    x, code, n, dev = _prep_input(tensor)
    q = torch.empty(tensor.shape, dtype=torch.uint8, device=dev)
    if n:
        with _host.device_guard(dev):
            st = _lib.lib().quanta_quantize_fp(x.data_ptr(), code, n, bits, q.data_ptr(), _host.stream_ptr(dev))
        _lib.check(st, "quanta_quantize_fp")
    return q, None, (1 if bits == 4 else 7)


def _dequantize_fp(q_tensor, bias, bits, out_dtype):
    q = _prep_codes(q_tensor)
    dev = q.device
    if float(bias) != int(bias):
        raise ValueError("the exponent bias must be an integer")
    out = torch.empty(q.shape, dtype=out_dtype, device=dev)
    if q.numel():
        with _host.device_guard(dev):
            st = _lib.lib().quanta_dequantize_fp(q.data_ptr(), q.numel(), bits, int(bias), out.data_ptr(),
                                                 _host._DTYPE[out_dtype], _host.stream_ptr(dev))
        _lib.check(st, "quanta_dequantize_fp")
    return out


def quantize_4bit(tensor, quant_type="linear", per_channel=False, blocksize=None, packed=False):
    """Quantize a floating-point tensor to 4-bit precision (codes 0..15, one per
    uint8 unless ``packed``).  Mirrors Quanta/functional/quantization.py:7-18."""
    if quant_type == "linear":
        return _quantize_linear(tensor, 4, per_channel, blocksize, packed)
    if quant_type == "nf4":
        # returns (indices, nf4_levels, abs_max) like the reference (:118)
        return _quantize_codebook(tensor, "nf4", blocksize, packed)
    if quant_type == "fp4":
        return _quantize_fp(tensor, 4)
    raise ValueError(f"Unknown quantization type: {quant_type}")


def quantize_8bit(tensor, quant_type="linear", per_channel=False, blocksize=None):
    """Quantize a floating-point tensor to 8-bit precision.
    Mirrors Quanta/functional/quantization.py:20-31."""
    if quant_type == "linear":
        return _quantize_linear(tensor, 8, per_channel, blocksize, False)
    if quant_type == "nf8":
        # returns (indices, nf8_levels, abs_max) like the reference (:183)
        return _quantize_codebook(tensor, "nf8", blocksize)
    if quant_type == "fp8":
        return _quantize_fp(tensor, 8)
    raise ValueError(f"Unknown quantization type: {quant_type}")


def _quantize_many(tensors, bits, blocksize, packed):
    import ctypes as C
    tensors = list(tensors)
    if not tensors:
        return []
    B = int(blocksize)
    dev = tensors[0].device
    xs, outs = [], []
    for t in tensors:
        _host.require_cuda(t)
        if t.device != dev or t.dtype != tensors[0].dtype:
            raise ValueError("all tensors of a batch must share one device and dtype")
        x = t.detach()
        if not x.is_contiguous():
            x = x.contiguous()
        n = x.numel()
        if n == 0 or n % B:
            raise ValueError(f"numel ({n}) must be a positive multiple of blocksize ({blocksize})")
        xs.append(x)
    code = _host.dtype_code(xs[0])
    with _host.device_guard(dev):
        for x in xs:
            n = x.numel()
            q = torch.empty((n + 1) // 2 if packed else n, dtype=torch.uint8, device=dev)
            outs.append((q, torch.empty(n // B, dtype=torch.float32, device=dev),
                         torch.empty(n // B, dtype=torch.float32, device=dev)))
        k = len(xs)
        arr = C.c_void_p * k
        st = _lib.lib().quanta_quantize_block_batch(
            arr(*[x.data_ptr() for x in xs]), (C.c_int64 * k)(*[x.numel() for x in xs]), k, code, B, bits,
            int(bool(packed)), arr(*[o[0].data_ptr() for o in outs]), arr(*[o[1].data_ptr() for o in outs]),
            arr(*[o[2].data_ptr() for o in outs]), _host.stream_ptr(dev))
    _lib.check(st, "quanta_quantize_block_batch")
    return [(q if packed else q.reshape(t.shape), s, z) for (q, s, z), t in zip(outs, tensors)]


def quantize_4bit_many(tensors, blocksize=64, packed=True):
    """Blockwise 4-bit quantization of many tensors in as few launches as possible — the fused form
    of the per-parameter loop in ``ModelQuantize.quantize`` (Quanta/functional/model.py:254-289).
    Returns ``[quantize_4bit(t, blocksize=blocksize, packed=packed) for t in tensors]`` (same bits)."""
    return _quantize_many(tensors, 4, blocksize, packed)


def quantize_8bit_many(tensors, blocksize=64):
    """Blockwise 8-bit twin of :func:`quantize_4bit_many`."""
    return _quantize_many(tensors, 8, blocksize, False)


def quantize_nf4_many(tensors, blocksize=64, packed=True):
    """NF4 twin of :func:`quantize_4bit_many` for a model of ``Linear4bit`` layers (default ``quant_type="nf4"``):
    ``[quantize_4bit(t, quant_type="nf4", blocksize=blocksize, packed=packed) for t in tensors]``.  One launch per
    tensor: the NF4 code search is latency-bound and its high-occupancy kernel measured faster than the
    multi-tensor TMA stream that serves the affine formats (46.6 vs 64.7 us on 11008 x 4096)."""
    return [_quantize_codebook(t, "nf4", blocksize, packed) for t in tensors]


def _dequantize_linear(q_tensor, scale, zero_point, blocksize, packed, shape, out_dtype):
    q = _prep_codes(q_tensor)
    dev = q.device
    scale = torch.as_tensor(scale, dtype=torch.float32, device=dev).contiguous()
    zp = torch.as_tensor(zero_point, dtype=torch.float32, device=dev).contiguous()
    out_shape = _out_shape(q, packed, shape)
    n = out_shape.numel()
    if n == 0:
        return torch.empty(out_shape, dtype=out_dtype, device=dev)
    ns = scale.numel()
    if zp.numel() != ns:
        if zp.numel() == 1:
            zp = zp.expand(ns).contiguous()
        elif ns == 1:
            scale = scale.expand(zp.numel()).contiguous()
            ns = zp.numel()
        else:
            raise ValueError("scale and zero_point must have the same number of elements")
    rows, cols = (out_shape[0], n // out_shape[0]) if len(out_shape) > 1 else (1, n)
    trailing = tuple(out_shape[1:])
    if blocksize is not None:
        B = int(blocksize)
        if B <= 0 or n % B or ns != n // B:
            raise ValueError("scale/zero_point do not match blocksize")
        mode = _lib.MODE_BLOCK
    elif ns == 1:
        mode, B = _lib.MODE_TENSOR, 0
    elif len(out_shape) > 1 and tuple(scale.shape) in ((1,) + trailing, trailing):
        # the reference just broadcasts ``q.float() * scale``: a per_channel scale [1, *shape[1:]]
        mode, B = _lib.MODE_DIM0, 0
    else:
        raise ValueError(f"scale of shape {tuple(scale.shape)} does not broadcast like the reference's per-tensor / "
                         f"per_channel results over codes of shape {tuple(out_shape)}; pass blocksize= for blockwise")
    out = torch.empty(out_shape, dtype=out_dtype, device=dev)
    with _host.device_guard(dev):
        st = _lib.lib().quanta_dequantize_affine(q.data_ptr(), int(bool(packed)), rows, cols, mode, B,
                                                 scale.data_ptr(), zp.data_ptr(), out.data_ptr(),
                                                 _host._DTYPE[out_dtype], _host.stream_ptr(dev))
    _lib.check(st, "quanta_dequantize_affine")
    return out


def _dequantize_many(qs, scales, zero_points, blocksize, packed, shapes, out_dtype):
    import ctypes as C
    qs, scales, zero_points = list(qs), list(scales), list(zero_points)
    if not (len(qs) == len(scales) == len(zero_points)):
        raise ValueError("qs, scales and zero_points must have the same length")
    if not qs:
        return []
    B = int(blocksize)
    if B <= 0 or B % 4:
        raise ValueError("blocksize must be a positive multiple of 4")
    if out_dtype not in _host._DTYPE:
        raise ValueError(f"unsupported out_dtype {out_dtype}")
    shapes = list(shapes) if shapes is not None else [None] * len(qs)
    dev = qs[0].device
    cq, cs, cz, ns, out_shapes = [], [], [], [], []
    for q, s, z, shape in zip(qs, scales, zero_points, shapes):
        q = _prep_codes(q)
        if q.device != dev:
            raise ValueError("all tensors of a batch must share one device")
        out_shape = _out_shape(q, packed, shape)
        n = out_shape.numel()
        if n == 0 or n % B:
            raise ValueError(f"numel ({n}) must be a positive multiple of blocksize ({blocksize})")
        s = torch.as_tensor(s, dtype=torch.float32, device=dev).contiguous()
        z = torch.as_tensor(z, dtype=torch.float32, device=dev).contiguous()
        if s.numel() != n // B or z.numel() != n // B:
            raise ValueError("scale/zero_point do not match blocksize")
        cq.append(q); cs.append(s); cz.append(z); ns.append(n); out_shapes.append(out_shape)
    with _host.device_guard(dev):
        outs = [torch.empty(sh, dtype=out_dtype, device=dev) for sh in out_shapes]
        k = len(cq)
        arr = C.c_void_p * k
        st = _lib.lib().quanta_dequantize_block_batch(
            arr(*[q.data_ptr() for q in cq]), (C.c_int64 * k)(*ns), k, int(bool(packed)), B,
            arr(*[s.data_ptr() for s in cs]), arr(*[z.data_ptr() for z in cz]), arr(*[o.data_ptr() for o in outs]),
            _host._DTYPE[out_dtype], _host.stream_ptr(dev))
    _lib.check(st, "quanta_dequantize_block_batch")
    return outs


def dequantize_4bit_many(qs, scales, zero_points, blocksize=64, packed=True, shapes=None, out_dtype=torch.float32):
    """Blockwise 4-bit dequantization of many tensors in as few launches as possible — the fused form of the
    per-tensor calls of ``QuantizationState.dequantize_tensor`` (Quanta/functional/state.py:246-281).  Returns
    ``[dequantize_4bit(q, s, z, blocksize=blocksize, packed=packed, shape=shape) for ...]`` (same bits)."""
    return _dequantize_many(qs, scales, zero_points, blocksize, packed, shapes, out_dtype)


def dequantize_8bit_many(qs, scales, zero_points, blocksize=64, out_dtype=torch.float32):
    """Blockwise 8-bit twin of :func:`dequantize_4bit_many`."""
    return _dequantize_many(qs, scales, zero_points, blocksize, False, None, out_dtype)


def dequantize_8bit(q_tensor, scale_or_levels, zero_point_or_bias, quant_type="linear", blocksize=None,
                    out_dtype=torch.float32):
    """Dequantize an 8-bit tensor back to floating point:
    ``q.float() * scale + zero_point`` (Quanta/functional/quantization.py:33-38)."""
    if quant_type == "linear":
        return _dequantize_linear(q_tensor, scale_or_levels, zero_point_or_bias, blocksize, False, None, out_dtype)
    if quant_type == "nf8":
        # scale_or_levels is the nf8_levels tensor, zero_point_or_bias the abs_max (:39-41)
        return _dequantize_codebook(q_tensor, zero_point_or_bias, "nf8", blocksize, False, None, out_dtype)
    if quant_type == "fp8":
        return _dequantize_fp(q_tensor, zero_point_or_bias, 8, out_dtype)
    raise ValueError(f"Unknown quantization type: {quant_type}")


def dequantize_4bit(q_tensor, scale_or_levels, zero_point_or_bias, quant_type="linear", blocksize=None,
                    packed=False, shape=None, out_dtype=torch.float32):
    """Dequantize a 4-bit tensor back to floating point
    (Quanta/functional/quantization.py:53-58).  ``packed=True`` takes the
    nibble-packed bytes of ``pack_4bit_tensor`` plus the original ``shape``."""
    if quant_type == "linear":
        return _dequantize_linear(q_tensor, scale_or_levels, zero_point_or_bias, blocksize, packed, shape, out_dtype)
    if quant_type == "nf4":
        # scale_or_levels is the nf4_levels tensor, zero_point_or_bias the abs_max (:59-61)
        return _dequantize_codebook(q_tensor, zero_point_or_bias, "nf4", blocksize, packed, shape, out_dtype)
    if quant_type == "fp4":
        return _dequantize_fp(q_tensor, zero_point_or_bias, 4, out_dtype)
    raise ValueError(f"Unknown quantization type: {quant_type}")
