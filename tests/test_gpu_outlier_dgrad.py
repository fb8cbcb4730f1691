"""GPU tests of the input gradient of the outlier-split Linear8bitLt: dx = dy . W16 with
W16[n, k] = round_act(qw[n, k] / cw[n]) (quanta_int8_outlier_dgrad, the int8 row-wise format of the
fused dequantize-transposed GEMM), and the autograd path of Linear8bitLt(outlier_split=True) built on it.

The oracle is dy.double() @ W16.double() on the CPU, with W16 computed on the CPU by an IEEE divide and
one rounding; the tolerance is that of test_gpu_gemm.py: 1e-2 of max|ref|."""

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
TOL = 1e-2


def rowwise_weight(N, K, seed, scale=0.02):
    from quanta_b200.nn import rowwise_quantize_sym
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(N, K, generator=g) * scale).cuda()
    return rowwise_quantize_sym(w)


def w16_ref(qw, cw, dtype):
    """round_act(qw / cw) on the CPU: an IEEE float32 divide, then one rounding to dtype."""
    return (qw.cpu().float() / cw.cpu()[:, None]).to(dtype)


def rel_err(a, ref):
    return float((a.double() - ref.double()).abs().max() / (ref.double().abs().max() + 1e-30))


def bits(t):
    return t.view(torch.int16)


# (N, K, M): N % 8 != 0 (1001), N % 64 != 0 (200, 1004); K = 64 * odd (320, 576), 16 * odd (80, 336, 4112)
# and 4096 / 16384; M from 1 to 2048 across the 16 / 64 / 256-row tiles
SHAPES = [(200, 320, 1), (1004, 336, 5), (1001, 4112, 16), (200, 80, 17), (1001, 576, 33), (1004, 4096, 256),
          (200, 16384, 300), (1001, 336, 2048)]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", SHAPES)
def test_outlier_dgrad_matches_oracle(dtype, shape):
    from quanta_b200.nn import int8_outlier_dgrad
    N, K, M = shape
    qw, cw = rowwise_weight(N, K, seed=N + K + M)
    g = torch.Generator().manual_seed(M)
    dy = torch.randn(M, N, generator=g).to(dtype)
    dx = int8_outlier_dgrad(dy.cuda(), qw, cw)
    assert dx.shape == (M, K) and dx.dtype == dtype
    ref = dy.double() @ w16_ref(qw, cw, dtype).double()
    err = rel_err(dx.cpu(), ref)
    assert err < TOL, f"rel err {err:.3e} {dtype} N={N} K={K} M={M}"


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("NK", [(1001, 336), (4096, 4096)])
def test_outlier_dgrad_weights_are_the_forwards(dtype, NK):
    """dy = I: dx is the weight matrix itself, and must be round_act(qw / cw) bit for bit, i.e. the weights
    of the forward's outlier columns and Linear8bitLt.dequantize_weight.  Degenerate rows take the true
    divide: all-zero and subnormal rows (cw = inf), a row of 1e-20 values (cw > 2^60) and a row holding one
    large value (cw < 2^-60 in bf16; within the fp16 range for fp16).  The subnormal row's codes are +-127,
    so its weights are +-0; a sum of products returns -0 as +0, so zeros are compared without their sign."""
    from quanta_b200.nn import Linear8bitLt, int8_outlier_dgrad
    N, K = NK
    g = torch.Generator().manual_seed(N + K)
    w = torch.randn(N, K, generator=g) * 0.02
    w[3] = 0.0
    w[N // 2] = torch.randn(K, generator=g) * 1e-40          # subnormal float32
    w[N // 3] = torch.randn(K, generator=g) * 1e-20
    w[N - 1, 5] = 3e38 if dtype == torch.bfloat16 else 6e4
    lin = Linear8bitLt(K, N, bias=False, outlier_split=True).cuda()
    lin.load_float_weight(w.cuda())
    qw, cw = lin.qweight_rowwise, lin.row_scale
    outside = ~((cw >= 2.0 ** -60) & (cw <= 2.0 ** 60))
    assert bool(outside[N // 3]) and (dtype != torch.bfloat16 or bool(outside[N - 1])), cw[[3, N // 2, N // 3, N - 1]]
    dx = int8_outlier_dgrad(torch.eye(N, device="cuda", dtype=dtype), qw, cw)
    ref = w16_ref(qw, cw, dtype)
    assert torch.isfinite(ref.float()).all()
    assert torch.equal(bits(dx.cpu()), bits(ref + 0.0))
    assert torch.equal(bits(dx), bits(lin.dequantize_weight(dtype) + 0.0))


@pytest.mark.parametrize("NK", [(4096, 4096), (16384, 4096), (4096, 16384)])
@pytest.mark.parametrize("M", [16, 256, 2048])
def test_outlier_dgrad_opt_shapes(NK, M):
    """OPT-6.7B shapes: a column slice against the float64 oracle, the whole output against an fp32 GEMM."""
    from quanta_b200.nn import int8_outlier_dgrad
    N, K = NK
    dtype = torch.bfloat16
    qw, cw = rowwise_weight(N, K, seed=N + M)
    w16 = (qw.float() / cw[:, None]).to(dtype)
    g = torch.Generator(device="cuda").manual_seed(M)
    dy = torch.randn(M, N, generator=g, device="cuda").to(dtype)
    dx = int8_outlier_dgrad(dy, qw, cw)
    cols = slice(K - 192, K)
    ref = dy.double().cpu() @ w16_ref(qw[:, cols], cw, dtype).double()
    err = rel_err(dx[:, cols].cpu(), ref)
    assert err < TOL, f"slice rel err {err:.3e}"
    err = rel_err(dx, dy.float() @ w16.float())
    assert err < TOL, f"full rel err {err:.3e}"


@pytest.mark.parametrize("shape", [(4096, 4096, 256), (1001, 4112, 16), (16384, 4096, 64)])
def test_outlier_dgrad_is_deterministic(shape):
    from quanta_b200.nn import int8_outlier_dgrad
    N, K, M = shape
    qw, cw = rowwise_weight(N, K, seed=7)
    dy = torch.randn(M, N, device="cuda").to(torch.bfloat16)
    a = int8_outlier_dgrad(dy, qw, cw)
    b = int8_outlier_dgrad(dy, qw, cw)
    assert torch.equal(bits(a), bits(b))


def test_outlier_dgrad_empty():
    from quanta_b200.nn import int8_outlier_dgrad
    qw, cw = rowwise_weight(64, 336, seed=1)
    dx = int8_outlier_dgrad(torch.empty(2, 0, 64, device="cuda", dtype=torch.bfloat16), qw, cw)
    assert dx.shape == (2, 0, 336)
    qw0, cw0 = qw[:0].contiguous(), cw[:0].contiguous()
    dx = int8_outlier_dgrad(torch.empty(3, 0, device="cuda", dtype=torch.float16), qw0, cw0)
    assert dx.shape == (3, 336) and not dx.any()


def outlier_layer(K, N, seed, bias=True):
    from quanta_b200.nn import Linear8bitLt
    torch.manual_seed(seed)
    lin = Linear8bitLt(K, N, bias=bias, outlier_split=True).cuda()
    lin.quantize_()
    return lin


def outlier_input(shape, K, dtype, seed):
    """Activations with a few feature columns far above the threshold 6, so the forward runs its 16-bit part."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(*shape, K, generator=g)
    x[..., [1, K // 3, K - 2]] *= 20.0
    return x.to(dtype).cuda()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("KNM", [(512, 1001, 3), (336, 1001, 64), (512, 200, 300)])
def test_layer_autograd_matches_float_twin(dtype, KNM):
    K, N, M = KNM
    lin = outlier_layer(K, N, seed=M)
    x = outlier_input((2, M), K, dtype, seed=M).requires_grad_(True)
    with torch.no_grad():
        y_ng = lin(x)
    y = lin(x)
    assert y.requires_grad
    assert torch.equal(bits(y.detach()), bits(y_ng)), "grad-enabled forward changed the output"
    dy = torch.randn_like(y)
    y.backward(dy)

    w16 = lin.dequantize_weight(dtype)
    x2 = x.detach().clone().requires_grad_(True)
    b2 = lin.bias.detach().clone().requires_grad_(True)
    F.linear(x2, w16, b2.to(dtype)).backward(dy)
    assert x.grad.dtype == dtype
    assert rel_err(x.grad, x2.grad) < TOL
    assert lin.bias.grad.dtype == lin.bias.dtype
    assert rel_err(lin.bias.grad, b2.grad) < TOL
    assert rel_err(lin.bias.grad, dy.reshape(-1, N).double().sum(0)) < 1e-3


def test_layer_bias_only_gradient():
    """x without requires_grad, bias trainable: only the bias gets a gradient."""
    lin = outlier_layer(256, 128, seed=1)
    x = outlier_input((8,), 256, torch.bfloat16, seed=1)
    lin(x).float().sum().backward()
    assert lin.bias.grad is not None and torch.allclose(lin.bias.grad, torch.full_like(lin.bias, 8.0))


def test_layer_float32_input():
    """fp32 x runs through the layer's fp16 compute dtype; x.grad comes back in fp32."""
    lin = outlier_layer(512, 384, seed=2)
    x = outlier_input((16,), 512, torch.float32, seed=2).requires_grad_(True)
    y = lin(x)
    assert y.dtype == torch.float32
    dy = torch.randn_like(y)
    y.backward(dy)
    x2 = x.detach().half().requires_grad_(True)
    F.linear(x2, lin.dequantize_weight(torch.float16), lin.bias.detach().half()).backward(dy.half())
    assert x.grad.dtype == torch.float32
    assert rel_err(x.grad, x2.grad) < TOL
    assert rel_err(lin.bias.grad, dy.double().sum(0)) < 1e-3


class LoraBlock(nn.Module):
    """Frozen outlier-split int8 base + trainable low-rank adapter: base(x) + (x A^T) B^T.  The twin keeps
    the base's forward values and takes its gradient from F.linear with the dequantized weight, so that
    only the backward differs between the two."""

    def __init__(self, base, r=8, seed=0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.base = base
        self.A = nn.Parameter((torch.randn(r, base.in_features, generator=g) * 0.05).to(torch.bfloat16).cuda())
        self.B = nn.Parameter((torch.randn(base.out_features, r, generator=g) * 0.05).to(torch.bfloat16).cuda())
        self.w16 = base.dequantize_weight(torch.bfloat16)

    def forward(self, x, twin=False):
        if twin:
            with torch.no_grad():
                y = self.base(x)
            lin = F.linear(x, self.w16, self.base.bias.to(torch.bfloat16))
            base = y + (lin - lin.detach())
        else:
            base = self.base(x)
        return base + (x @ self.A.t()) @ self.B.t()


def lora_stack():
    blocks = nn.ModuleList([LoraBlock(outlier_layer(512, 512, seed=i), seed=i) for i in range(2)])
    for b in blocks:
        b.base.bias.requires_grad_(False)
    return blocks


def run_stack(blocks, x, twin=False):
    h = x
    for b in blocks:
        h = b(h, twin)
    return h.float().square().sum()


def test_int8_lora_lower_adapter_gradients():
    """Two stacked outlier-split layers with adapters: the lower adapters' gradients need the upper base's dy @ W."""
    blocks = lora_stack()
    x = outlier_input((64,), 512, torch.bfloat16, seed=3)
    run_stack(blocks, x).backward()
    got = [p.grad.clone() for p in (blocks[0].A, blocks[0].B)]
    for b in blocks:
        b.A.grad = b.B.grad = None
    run_stack(blocks, x, twin=True).backward()
    want = [p.grad for p in (blocks[0].A, blocks[0].B)]
    for g, w in zip(got, want):
        assert rel_err(g, w) < 2 * TOL


def test_int8_lora_graph_capture_is_bit_identical():
    blocks = lora_stack()
    params = [p for b in blocks for p in (b.A, b.B)]
    x = outlier_input((64,), 512, torch.bfloat16, seed=4)

    def step():
        for p in params:
            p.grad = None
        loss = run_stack(blocks, x)
        loss.backward()
        return loss

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    for p in params:
        p.grad = None
    with torch.cuda.graph(graph):
        loss_g = run_stack(blocks, x)
        loss_g.backward()
    graph.replay()
    torch.cuda.synchronize()
    replayed = [p.grad.clone() for p in params]
    loss_e = step()
    torch.cuda.synchronize()
    assert torch.equal(loss_g, loss_e)
    for g, e in zip(replayed, [p.grad for p in params]):
        assert torch.equal(bits(g), bits(e))
