"""Drop-in CUDA versions of ``Quanta.nn.Linear8bitLt`` / ``Linear4bit``.

Constructor signatures and attributes are those of the reference
(Quanta/nn/linear.py:14-21, :52-59).  The reference's ``forward`` is a
placeholder ``F.linear(x, self.weight, self.bias)`` on floating-point weights
(:43-45, :81-83); here the weight is held quantized (convention A, blockwise
along in_features) and ``forward`` is the fused dequantize-then-matmul kernel:

    y = x @ dequantize_*bit(Wq, scale, zero_point).to(x.dtype).T + bias

Parity: defined by that composition (SURVEY §8(c)); tolerance 1e-2 relative in
bf16/fp16.  ``Linear4bit`` supports ``quant_type="nf4"`` (the reference default: NF4 codebook,
blockwise abs_max) and ``quant_type="linear"`` (blockwise affine).

Backward: the quantized weight is frozen (its codes are buffers).  When autograd is recording and x or
the bias requires a gradient, ``Linear4bit`` and ``Linear8bitLt`` run through an autograd Function whose
backward gives ``x.grad = dy @ W`` (the fused dequantize-transposed GEMM, with bit-for-bit the weights of
the forward) and ``bias.grad = dy.sum(0)`` (fp32 accumulation).  The forward launches the same kernel with
the same arguments either way.  With ``outlier_split=True`` the gradient is the straight-through one of
the LLM.int8() product (bitsandbytes' ``MatMul8bitLt``): W is ``dequantize_weight(dtype)``, i.e.
``round_act(qw / row_scale)``, and the threshold, the outlier columns and the int8 quantization of x do
not enter.  Not differentiable: the tensor-parallel layers, the weight itself, and a double backward.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from ..functional.quantization import quantize_4bit, quantize_8bit, dequantize_4bit, dequantize_8bit
from .functional import (linear_wna16, linear_nf4a16, int8_outlier_matmul, rowwise_quantize_sym, LinearWNA16Function,
                         LinearNF4A16Function, Int8OutlierMatmulFunction)


_QUANT_BUFFERS = ("qweight", "scale", "zero_point", "qweight_rowwise", "row_scale")
_FLOAT32_BUFFERS = ("scale", "zero_point", "row_scale")


class _QuantLinearBase(nn.Module):
    bits = 8

    # ---- the quantization parameters are float32 whatever the module is cast to -------------------
    def _apply(self, fn, *args, **kwargs):
        """``module.half()`` / ``.to(torch.bfloat16)`` cast every floating-point buffer; the kernels read
        scale / zero_point / row_scale as float32, so they are cast back (device moves are kept)."""
        out = super()._apply(fn, *args, **kwargs)
        for name in _FLOAT32_BUFFERS:
            buf = getattr(self, name, None)
            if isinstance(buf, torch.Tensor) and buf.dtype != torch.float32:
                setattr(self, name, buf.to(torch.float32))
        return out

    # ---- checkpoints: a quantized layer saves and reloads through state_dict ------------------------
    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        """A fresh module registers the quantized buffers as None and owns a full-size float weight; a quantized
        checkpoint holds the buffers and an empty weight.  Materialise whatever the checkpoint carries before the
        stock loader copies it in (which then sees matching shapes)."""
        quantized = False
        for name in _QUANT_BUFFERS:
            key = prefix + name
            if key in state_dict and name in self._buffers:
                src = state_dict[key]
                cur = self._buffers[name]
                if cur is None or cur.shape != src.shape or cur.dtype != src.dtype:
                    dev = self.weight.device if self.weight.numel() else (cur.device if cur is not None else src.device)
                    self._buffers[name] = torch.empty(src.shape, dtype=src.dtype, device=dev)
                quantized = True
        wkey = prefix + "weight"
        if wkey in state_dict and state_dict[wkey].shape != self.weight.shape:
            w = state_dict[wkey]
            if quantized and w.numel() == 0:        # quantized checkpoint: the float weight is gone
                self.weight = nn.Parameter(torch.empty(0, device=self.weight.device, dtype=w.dtype), requires_grad=False)
            elif w.dim() == 2 and tuple(w.shape) == (self.out_features, self.in_features):
                # float checkpoint into a module that was already quantized: take the weight, drop the stale codes
                self.weight = nn.Parameter(torch.empty_like(w, device=self.weight.device), requires_grad=False)
                for name in _QUANT_BUFFERS:
                    if name in self._buffers and prefix + name not in state_dict:
                        self._buffers[name] = None
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)

    def _init_common(self, in_features, out_features, bias, blocksize):
        self.in_features = in_features
        self.out_features = out_features
        self.blocksize = blocksize
        # like the reference, the module is born with a floating-point weight ...
        self.weight = nn.Parameter(torch.empty((out_features, in_features)))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_features))
        else:
            self.register_parameter("bias", None)
        # ... and holds the quantized form once quantize_() / load_float_weight() ran
        self.register_buffer("qweight", None, persistent=True)
        self.register_buffer("scale", None, persistent=True)
        self.register_buffer("zero_point", None, persistent=True)
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            fan_in, _ = nn.init._calculate_fan_in_and_fan_out(self.weight)
            bound = 1 / math.sqrt(fan_in) if fan_in > 0 else 0
            nn.init.uniform_(self.bias, -bound, bound)

    # ---- quantized state -------------------------------------------------
    def _check_quant_type(self):
        pass

    @torch.no_grad()
    def quantize_(self):
        """Quantize the current floating-point weight on its (CUDA) device and drop it."""
        self._check_quant_type()
        w = self.weight.detach()
        if self.in_features % self.blocksize:
            raise ValueError(f"in_features ({self.in_features}) must be a multiple of blocksize ({self.blocksize})")
        if self.bits == 4:
            q, s, z = quantize_4bit(w, blocksize=self.blocksize, packed=True)
        else:
            q, s, z = quantize_8bit(w, blocksize=self.blocksize)
        self.qweight, self.scale, self.zero_point = q, s, z
        self.weight = nn.Parameter(torch.empty(0, device=w.device), requires_grad=False)
        return self

    @torch.no_grad()
    def load_float_weight(self, weight, bias=None):
        """Install a floating-point [out, in] weight (and bias) and quantize it."""
        if tuple(weight.shape) != (self.out_features, self.in_features):
            raise ValueError("weight shape mismatch")
        self.weight = nn.Parameter(weight.detach().clone(), requires_grad=False)
        if bias is not None and self.bias is not None:
            self.bias.data = bias.detach().to(self.bias.dtype).clone()
        return self.quantize_()

    def dequantize_weight(self, dtype=torch.float32):
        """The [out, in] floating-point weight the forward pass multiplies with."""
        shape = (self.out_features, self.in_features)
        if self.bits == 4:
            return dequantize_4bit(self.qweight, self.scale, self.zero_point, blocksize=self.blocksize, packed=True,
                                   shape=shape, out_dtype=dtype)
        return dequantize_8bit(self.qweight.reshape(shape), self.scale, self.zero_point, blocksize=self.blocksize,
                               out_dtype=dtype)

    def _bias_as(self, dtype, device):
        """The bias in the compute dtype, converted once per (dtype, device, bias version) instead of on every forward."""
        b = self.bias
        if b is None:
            return None
        if b.dtype == dtype and b.device == device and b.is_contiguous():
            return b
        key = (dtype, device, b._version, b.data_ptr())
        cache = self.__dict__.get("_bias_cache")
        if cache is None or cache[0] != key:
            cache = (key, b.detach().to(device=device, dtype=dtype).contiguous())
            self.__dict__["_bias_cache"] = cache
        return cache[1]

    def _forward_quantized(self, x, compute_dtype):
        if self.qweight is None:
            if not self.weight.is_cuda:
                raise RuntimeError("quanta_b200 layers run on CUDA only: move the module to a GPU first")
            self.quantize_()
        xin = x if x.dtype == compute_dtype else x.to(compute_dtype)
        if self._records_grad(xin):
            y = LinearWNA16Function.apply(xin, self.bias, self._bias_as(compute_dtype, x.device), self.qweight, self.scale,
                                          self.zero_point, self.bits, self.blocksize, self.out_features, self.in_features)
        else:
            y = linear_wna16(xin, self.qweight, self.scale, self.zero_point, self._bias_as(compute_dtype, x.device),
                             bits=self.bits, blocksize=self.blocksize, out_features=self.out_features,
                             in_features=self.in_features)
        return y if y.dtype == x.dtype or not x.is_floating_point() else y.to(x.dtype)

    def _records_grad(self, x):
        """Whether autograd needs this call: grad mode on and x or the bias requires a gradient."""
        return torch.is_grad_enabled() and (x.requires_grad or (self.bias is not None and self.bias.requires_grad))


class Linear8bitLt(_QuantLinearBase):
    """8-bit quantized linear layer (Quanta/nn/linear.py:10-45).

    ``outlier_split=False`` (default): blockwise W8A16 dequant-GEMM (row G2).
    ``outlier_split=True``: the LLM.int8() decomposition the reference's
    ``threshold`` argument points at (row G3) — row-wise symmetric int8 weight
    codes, int8 x int8 tensor-core product for the regular feature columns and
    a 16-bit product for the columns whose activations exceed ``threshold``.

    Differentiable in x and bias in both modes (module docstring).  With ``outlier_split=True`` the
    backward is straight-through: ``x.grad = dy @ dequantize_weight(dtype)``, the 16-bit weights the
    forward uses for its outlier columns, whatever the threshold selected; the 8-bit LoRA setting of a
    frozen int8 base under trainable adapters gets the base's ``dy @ W`` term in ``x.grad``."""
    bits = 8

    def __init__(self, in_features, out_features, bias=True, has_fp16_weights=False, threshold=6.0, blocksize=64,
                 outlier_split=False):
        super().__init__()
        self.threshold = threshold
        self.has_fp16_weights = has_fp16_weights
        self.outlier_split = outlier_split
        self._init_common(in_features, out_features, bias, blocksize)
        self.register_buffer("qweight_rowwise", None, persistent=True)
        self.register_buffer("row_scale", None, persistent=True)

    @torch.no_grad()
    def quantize_(self):
        if not self.outlier_split:
            return super().quantize_()
        w = self.weight.detach()
        self.qweight_rowwise, self.row_scale = rowwise_quantize_sym(w)
        self.weight = nn.Parameter(torch.empty(0, device=w.device), requires_grad=False)
        return self

    def dequantize_weight(self, dtype=torch.float32):
        if not self.outlier_split:
            return super().dequantize_weight(dtype)
        return (self.qweight_rowwise.float() / self.row_scale[:, None]).to(dtype)

    def forward(self, x):
        dt = x.dtype if x.dtype in (torch.float16, torch.bfloat16) else torch.float16
        if not self.outlier_split:
            return self._forward_quantized(x, dt)
        if self.qweight_rowwise is None:
            if not self.weight.is_cuda:
                raise RuntimeError("quanta_b200 layers run on CUDA only: move the module to a GPU first")
            self.quantize_()
        xin = x if x.dtype == dt else x.to(dt)
        if self._records_grad(xin):
            y = Int8OutlierMatmulFunction.apply(xin, self.bias, self._bias_as(dt, x.device), self.qweight_rowwise,
                                                self.row_scale, self.threshold)
        else:
            y = int8_outlier_matmul(xin, self.qweight_rowwise, self.row_scale, self.threshold, self._bias_as(dt, x.device))
        return y if y.dtype == x.dtype or not x.is_floating_point() else y.to(x.dtype)


class Linear4bit(_QuantLinearBase):
    """4-bit quantized linear layer (Quanta/nn/linear.py:48-83).

    ``quant_type="nf4"`` (the reference default): NF4 codebook with one abs_max per block of
    ``blocksize`` input features; ``quant_type="linear"``: blockwise affine min-max (convention A).
    Both are differentiable in x and bias (module docstring): the QLoRA setting of a frozen NF4 base
    under trainable adapters gets the base's ``dy @ W`` term in ``x.grad``."""
    bits = 4

    def __init__(self, in_features, out_features, bias=True, compute_dtype=torch.float16, quant_type="nf4",
                 blocksize=64):
        super().__init__()
        self.compute_dtype = compute_dtype
        self.quant_type = quant_type
        self._init_common(in_features, out_features, bias, blocksize)

    def _check_quant_type(self):
        if self.quant_type not in ("linear", "nf4"):
            raise NotImplementedError(f"quant_type={self.quant_type!r}: only 'nf4' and 'linear' have a fused dequant-GEMM; "
                                      "fp4 is available as quantize_4bit / dequantize_4bit (SURVEY §8(f) N4)")

    @torch.no_grad()
    def quantize_(self):
        if self.quant_type != "nf4":
            return super().quantize_()
        w = self.weight.detach()
        if self.in_features % self.blocksize:
            raise ValueError(f"in_features ({self.in_features}) must be a multiple of blocksize ({self.blocksize})")
        # scale holds abs_max per block; there is no zero-point
        self.qweight, _, self.scale = quantize_4bit(w, quant_type="nf4", blocksize=self.blocksize, packed=True)
        self.zero_point = None
        self.weight = nn.Parameter(torch.empty(0, device=w.device), requires_grad=False)
        return self

    def dequantize_weight(self, dtype=torch.float32):
        if self.quant_type != "nf4":
            return super().dequantize_weight(dtype)
        return dequantize_4bit(self.qweight, None, self.scale, quant_type="nf4", blocksize=self.blocksize, packed=True,
                               shape=(self.out_features, self.in_features), out_dtype=dtype)

    def forward(self, x):
        if self.quant_type != "nf4":
            self._check_quant_type()
            return self._forward_quantized(x, self.compute_dtype)
        if self.qweight is None:
            if not self.weight.is_cuda:
                raise RuntimeError("quanta_b200 layers run on CUDA only: move the module to a GPU first")
            self.quantize_()
        xin = x if x.dtype == self.compute_dtype else x.to(self.compute_dtype)
        if self._records_grad(xin):
            y = LinearNF4A16Function.apply(xin, self.bias, self._bias_as(self.compute_dtype, x.device), self.qweight,
                                           self.scale, self.blocksize, self.out_features, self.in_features)
        else:
            y = linear_nf4a16(xin, self.qweight, self.scale, self._bias_as(self.compute_dtype, x.device),
                              blocksize=self.blocksize, out_features=self.out_features, in_features=self.in_features)
        return y if y.dtype == x.dtype or not x.is_floating_point() else y.to(x.dtype)
