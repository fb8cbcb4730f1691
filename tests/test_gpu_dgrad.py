"""GPU tests of the input gradient of the quantized linear layers: dx = dy . dequant(Wq), the fused
dequantize-transposed GEMM (quanta_gemm_wna16_dgrad / quanta_gemm_nf4a16_dgrad), and the autograd path
of Linear4bit / Linear8bitLt built on it.

The oracle is dy.double() @ dequantize(q).to(dtype).double() on the CPU, with the library's bit-exact
dequantize; the tolerance is that of test_gpu_gemm.py: 1e-2 of max|ref|."""

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
TOL = 1e-2


def quantized_weight(fmt, N, K, blocksize, seed):
    """(codes, params) of a random [N, K] weight in format fmt (4, 8 or 'nf4'), and its 16-bit-ready
    float32 dequantization."""
    import quanta_b200 as Q
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(N, K, generator=g) * 0.02).cuda()
    if fmt == "nf4":
        q, _, absmax = Q.quantize_4bit(w, quant_type="nf4", blocksize=blocksize, packed=True)
        wd = Q.dequantize_4bit(q, None, absmax, quant_type="nf4", blocksize=blocksize, packed=True, shape=(N, K))
        return q, (absmax,), wd
    if fmt == 4:
        q, s, z = Q.quantize_4bit(w, blocksize=blocksize, packed=True)
        wd = Q.dequantize_4bit(q, s, z, blocksize=blocksize, packed=True, shape=(N, K))
    else:
        q, s, z = Q.quantize_8bit(w, blocksize=blocksize)
        wd = Q.dequantize_8bit(q.reshape(N, K), s, z, blocksize=blocksize)
    return q, (s, z), wd


def dgrad(fmt, dy, q, params, blocksize, N, K):
    from quanta_b200.nn import linear_wna16_dgrad, linear_nf4a16_dgrad
    if fmt == "nf4":
        return linear_nf4a16_dgrad(dy, q, params[0], blocksize=blocksize, out_features=N, in_features=K)
    return linear_wna16_dgrad(dy, q, params[0], params[1], bits=fmt, blocksize=blocksize, out_features=N, in_features=K)


def rel_err(a, ref):
    return float((a.double() - ref.double()).abs().max() / (ref.double().abs().max() + 1e-30))


def check_case(fmt, dtype, blocksize, N, K, M, seed):
    q, params, wd = quantized_weight(fmt, N, K, blocksize, seed)
    g = torch.Generator().manual_seed(seed + 1)
    dy = torch.randn(M, N, generator=g).to(dtype)
    dx = dgrad(fmt, dy.cuda(), q, params, blocksize, N, K)
    assert dx.shape == (M, K) and dx.dtype == dtype
    ref = dy.double() @ wd.to(dtype).double().cpu()
    err = rel_err(dx.cpu(), ref)
    assert err < TOL, f"rel err {err:.3e} fmt={fmt} {dtype} block={blocksize} N={N} K={K} M={M}"


SHAPES = [(200, 320, 1), (1004, 512, 5), (1001, 256, 16), (256, 4160, 17), (1001, 320, 33), (200, 1024, 256),
          (1004, 640, 300), (384, 4160, 2048)]


@pytest.mark.parametrize("fmt", [4, 8, "nf4"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", SHAPES)
def test_dgrad_matches_oracle(fmt, dtype, shape):
    N, K, M = shape
    check_case(fmt, dtype, 64, N, K, M, seed=N + K + M)


@pytest.mark.parametrize("fmt", [4, 8, "nf4"])
@pytest.mark.parametrize("blocksize", [128, 256])
@pytest.mark.parametrize("shape", [(1001, 512, 33), (200, 1024, 256), (96, 768, 7)])
def test_dgrad_blocksizes(fmt, blocksize, shape):
    N, K, M = shape
    check_case(fmt, torch.bfloat16, blocksize, N, K, M, seed=N + K + M + blocksize)


@pytest.mark.parametrize("fmt", [4, 8, "nf4"])
@pytest.mark.parametrize("NK", [(4096, 14336), (14336, 4096)])
@pytest.mark.parametrize("M", [16, 256, 2048])
def test_dgrad_llama3_8b_shapes(fmt, NK, M):
    """Llama-3-8B MLP shapes: a column slice against the float64 oracle, the whole output against an fp32 GEMM."""
    N, K = NK
    dtype = torch.bfloat16
    q, params, wd = quantized_weight(fmt, N, K, 64, seed=N + M)
    w16 = wd.to(dtype)
    g = torch.Generator(device="cuda").manual_seed(M)
    dy = torch.randn(M, N, generator=g, device="cuda").to(dtype)
    dx = dgrad(fmt, dy, q, params, 64, N, K)
    cols = slice(K - 192, K)
    ref = dy.double().cpu() @ w16[:, cols].double().cpu()
    err = rel_err(dx[:, cols].cpu(), ref)
    assert err < TOL, f"slice rel err {err:.3e}"
    full = dy.float() @ w16.float()
    err = rel_err(dx, full)
    assert err < TOL, f"full rel err {err:.3e}"


@pytest.mark.parametrize("fmt", [4, 8, "nf4"])
@pytest.mark.parametrize("shape", [(4096, 4096, 256), (1001, 4160, 16), (14336, 4096, 64)])
def test_dgrad_is_deterministic(fmt, shape):
    """Stream-K partial sums are reduced in a fixed order: two calls give the same bits."""
    N, K, M = shape
    q, params, _ = quantized_weight(fmt, N, K, 64, seed=7)
    dy = torch.randn(M, N, device="cuda").to(torch.bfloat16)
    a = dgrad(fmt, dy, q, params, 64, N, K)
    b = dgrad(fmt, dy, q, params, 64, N, K)
    assert torch.equal(a.view(torch.int16), b.view(torch.int16))


def make_layer(kind, K, N, seed):
    from quanta_b200.nn import Linear4bit, Linear8bitLt
    torch.manual_seed(seed)
    if kind == "nf4":
        lin = Linear4bit(K, N, bias=True, compute_dtype=torch.bfloat16, quant_type="nf4")
    elif kind == "linear4":
        lin = Linear4bit(K, N, bias=True, compute_dtype=torch.bfloat16, quant_type="linear")
    else:
        lin = Linear8bitLt(K, N, bias=True)
    lin = lin.cuda()
    lin.quantize_()
    return lin


@pytest.mark.parametrize("kind", ["nf4", "linear4", "int8"])
@pytest.mark.parametrize("M", [3, 64, 300])
def test_layer_autograd_matches_float_twin(kind, M):
    K, N = 512, 1001
    lin = make_layer(kind, K, N, seed=M)
    x = (torch.randn(2, M, K, device="cuda") * 0.5).to(torch.bfloat16).requires_grad_(True)
    with torch.no_grad():
        y_ng = lin(x)
    y = lin(x)
    assert y.requires_grad
    assert torch.equal(y.detach().view(torch.int16), y_ng.view(torch.int16)), "grad-enabled forward changed the output"
    dy = torch.randn_like(y)
    y.backward(dy)

    w16 = lin.dequantize_weight(torch.bfloat16)
    x2 = x.detach().clone().requires_grad_(True)
    b2 = lin.bias.detach().clone().requires_grad_(True)
    F.linear(x2, w16, b2.to(torch.bfloat16)).backward(dy)
    assert rel_err(x.grad, x2.grad) < TOL
    assert lin.bias.grad.dtype == lin.bias.dtype
    assert rel_err(lin.bias.grad, b2.grad) < TOL
    ref_db = dy.reshape(-1, N).double().sum(0)
    assert rel_err(lin.bias.grad, ref_db) < 1e-3


def test_layer_bias_only_gradient():
    """x without requires_grad, bias trainable: only the bias gets a gradient."""
    lin = make_layer("nf4", 256, 128, seed=1)
    x = torch.randn(8, 256, device="cuda").to(torch.bfloat16)
    lin(x).float().sum().backward()
    assert lin.bias.grad is not None and torch.allclose(lin.bias.grad, torch.full_like(lin.bias, 8.0))


class LoraBlock(nn.Module):
    """Frozen quantized base + trainable low-rank adapter: base(x) + (x A^T) B^T."""

    def __init__(self, base, r=8, seed=0):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.base = base
        self.A = nn.Parameter((torch.randn(r, base.in_features, generator=g) * 0.05).to(torch.bfloat16).cuda())
        self.B = nn.Parameter((torch.randn(base.out_features, r, generator=g) * 0.05).to(torch.bfloat16).cuda())
        self.w16 = None

    def forward(self, x, twin=False):
        if twin:
            base = F.linear(x, self.w16, self.base.bias.to(torch.bfloat16))
        else:
            base = self.base(x)
        return base + (x @ self.A.t()) @ self.B.t()


def qlora_stack():
    blocks = nn.ModuleList([LoraBlock(make_layer("nf4", 512, 512, seed=i), seed=i) for i in range(2)])
    for b in blocks:
        b.base.bias.requires_grad_(False)
        b.w16 = b.base.dequantize_weight(torch.bfloat16)
    return blocks


def run_stack(blocks, x, twin=False):
    h = x
    for b in blocks:
        h = b(h, twin)
    return h.float().square().sum()


def test_qlora_lower_adapter_gradients():
    """Two stacked NF4 layers with adapters: the lower adapters' gradients need the upper base's dy @ W."""
    blocks = qlora_stack()
    x = (torch.randn(64, 512, device="cuda")).to(torch.bfloat16)
    run_stack(blocks, x).backward()
    got = [p.grad.clone() for p in (blocks[0].A, blocks[0].B)]
    for b in blocks:
        b.A.grad = b.B.grad = None
    run_stack(blocks, x, twin=True).backward()
    want = [p.grad for p in (blocks[0].A, blocks[0].B)]
    for g, w in zip(got, want):
        assert rel_err(g, w) < 2 * TOL


def test_qlora_graph_capture_is_bit_identical():
    blocks = qlora_stack()
    params = [p for b in blocks for p in (b.A, b.B)]
    x = torch.randn(64, 512, device="cuda").to(torch.bfloat16)

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
        assert torch.equal(g.view(torch.int16), e.view(torch.int16))
