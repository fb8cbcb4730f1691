"""GPU tests of the fused dequantize-then-matmul (rows G1/G2).  The oracle is
the composition the reference's layers imply: F.linear(x, dequantize(q).to(x.dtype))
evaluated in float64 on the CPU (oracle.linear_dequant).  Tolerance (north_star):
1e-2 relative in bf16 — measured as max|y - ref| / max|ref|."""

import numpy as np
import pytest
import torch

from oracle import oracle_c as OC
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu
TOL = 1e-2


def make_case(N, K, M, bits, dtype, seed, bias=True):
    import quanta_b200 as Q
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(N, K, generator=g) * 0.02
    x = torch.randn(M, K, generator=g).to(dtype)
    b = (torch.randn(N, generator=g) * 0.1).to(dtype) if bias else None
    wd = w.cuda()
    if bits == 4:
        q, s, z = Q.quantize_4bit(wd, blocksize=64, packed=True)
    else:
        q, s, z = Q.quantize_8bit(wd, blocksize=64)
    return w, x, b, q, s, z


def reference(x, q, s, z, b, bits, N, K, dtype):
    """float64 composition oracle on the codes the GPU produced (codes themselves are
    checked bit-exactly in test_gpu_quantize.py)."""
    name = "bf16" if dtype == torch.bfloat16 else "fp16"
    xf = x.float().numpy()
    wq = q.cpu().numpy()
    if name == "bf16":
        return OC.linear_dequant(xf, wq, s.cpu().numpy(), z.cpu().numpy(), None if b is None else b.float().numpy(),
                                 bits, N, K, 64)
    codes = O.unpack4(wq)[: N * K].reshape(N, K) if bits == 4 else wq.reshape(N, K)
    return O.linear_dequant(xf, codes, s.cpu().numpy(), z.cpu().numpy(), None if b is None else b.float().numpy(), 64, name)


def rel_err(y, ref):
    return float(np.abs(y - ref).max() / (np.abs(ref).max() + 1e-30))


@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(128, 64, 1), (128, 256, 16), (256, 512, 5), (384, 1024, 33), (1024, 4096, 64),
                                   (200, 320, 7), (512, 2048, 256), (256, 1024, 300), (1004, 512, 48)])
def test_gemm_matches_composition_oracle(bits, dtype, shape):
    from quanta_b200.nn import linear_wna16
    N, K, M = shape
    w, x, b, q, s, z = make_case(N, K, M, bits, dtype, seed=N + K + M + bits)
    y = linear_wna16(x.cuda(), q, s, z, b.cuda(), bits=bits, blocksize=64, out_features=N)
    assert y.shape == (M, N) and y.dtype == dtype
    ref = reference(x, q, s, z, b, bits, N, K, dtype)
    err = rel_err(y.float().cpu().numpy(), ref)
    assert err < TOL, f"rel err {err:.3e} for N={N} K={K} M={M} bits={bits} {dtype}"


@pytest.mark.parametrize("bits", [4, 8])
def test_gemm_llama3_8b_shapes(bits):
    """Config 3: (N,K) in {(4096,14336),(14336,4096)}, M in 1..256 (subset), bf16."""
    from quanta_b200.nn import linear_wna16
    for (N, K) in ((4096, 14336), (14336, 4096)):
        w, x, b, q, s, z = make_case(N, K, 256, bits, torch.bfloat16, seed=N + bits, bias=False)
        xd = x.cuda()
        for M in (1, 16, 64, 256):
            y = linear_wna16(xd[:M], q, s, z, None, bits=bits, blocksize=64, out_features=N)
            # oracle on a slice of output features to keep the CPU time bounded
            cols = slice(0, 256)
            nb = K // 64
            ref = OC.linear_dequant(x[:M].float().numpy(),
                                    q.cpu().numpy().reshape(N, -1)[cols], s.cpu().numpy().reshape(N, nb)[cols],
                                    z.cpu().numpy().reshape(N, nb)[cols], None, bits, 256, K, 64)
            err = rel_err(y[:, cols].float().cpu().numpy(), ref)
            assert err < TOL, f"rel err {err:.3e} N={N} K={K} M={M} bits={bits}"
            # full-size property: against torch matmul with the GPU-dequantized weight (same rounding to bf16)
            from quanta_b200 import dequantize_4bit, dequantize_8bit
            wd = (dequantize_4bit(q, s, z, blocksize=64, packed=True, shape=(N, K), out_dtype=torch.bfloat16) if bits == 4
                  else dequantize_8bit(q.reshape(N, K), s, z, blocksize=64, out_dtype=torch.bfloat16))
            yt = (xd[:M].float() @ wd.float().t())
            e2 = float((y.float() - yt).abs().max() / yt.abs().max())
            assert e2 < TOL, f"vs torch fp32 matmul: {e2:.3e}"


@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("blocksize", [128, 256])
def test_gemm_larger_blocksizes(bits, blocksize):
    """block = 64 * 2^j: one scale per `blocksize` K values (scalar parameter path of the kernel)."""
    import quanta_b200 as Q
    from quanta_b200.nn import linear_wna16
    N, K, M = 384, 1024, 40
    g = torch.Generator().manual_seed(blocksize + bits)
    w = torch.randn(N, K, generator=g) * 0.02
    x = torch.randn(M, K, generator=g).to(torch.bfloat16)
    if bits == 4:
        q, s, z = Q.quantize_4bit(w.cuda(), blocksize=blocksize, packed=True)
        codes = O.unpack4(q.cpu().numpy())[: N * K].reshape(N, K)
    else:
        q, s, z = Q.quantize_8bit(w.cuda(), blocksize=blocksize)
        codes = q.cpu().numpy().reshape(N, K)
    y = linear_wna16(x.cuda(), q, s, z, None, bits=bits, blocksize=blocksize, out_features=N)
    ref = O.linear_dequant(x.float().numpy(), codes, s.cpu().numpy(), z.cpu().numpy(), None, blocksize, "bf16")
    assert rel_err(y.float().cpu().numpy(), ref) < TOL


@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(128, 256, 1), (200, 512, 7), (136, 1536, 9), (384, 2048, 16), (1000, 4096, 3),
                                   (256, 6144, 12), (128, 8192, 8), (264, 768, 5), (300, 1280, 16), (512, 11008, 2)])
def test_small_batch_kernel(bits, dtype, shape):
    """M <= 16, K % 256 == 0 takes the weight-stream kernel (csrc/gemm_small.cu): one and several K ranges per
    row tile (partials + last-arriver reduction), ragged N, batch rows past M zero-filled, and — 4-bit stages span
    512 K values — K that ends in the middle of a stage (256, 768, 1280, 11008: the tail is zero-filled)."""
    from quanta_b200.nn import linear_wna16
    N, K, M = shape
    w, x, b, q, s, z = make_case(N, K, M, bits, dtype, seed=3 * N + K + M + bits)
    xd, bd = x.cuda(), b.cuda()
    y = linear_wna16(xd, q, s, z, bd, bits=bits, blocksize=64, out_features=N)
    ref = reference(x, q, s, z, b, bits, N, K, dtype)
    err = rel_err(y.float().cpu().numpy(), ref)
    assert err < TOL, f"rel err {err:.3e} for N={N} K={K} M={M} bits={bits} {dtype}"
    # the exact-weight products put it well inside the tolerance: the only roundings are x and the output
    assert err < 4e-3
    for _ in range(3):                     # deterministic, counters left clean
        assert torch.equal(linear_wna16(xd, q, s, z, bd, bits=bits, blocksize=64, out_features=N), y)


@pytest.mark.parametrize("bits", [4, 8])
def test_gemm_right_behind_the_kernel_that_wrote_its_weights(bits):
    """The GEMM kernels are launched with programmatic stream serialization and start streaming their WEIGHTS before
    their dependency wait.  That is sound only because the kernels that write codes / scales never release their
    dependents early (common.cuh, pdl_wait): quantize fresh weights and multiply right behind, no synchronisation
    in between, many times; every result must equal the one computed after a device synchronise."""
    import quanta_b200 as Q
    from quanta_b200.nn import linear_wna16
    N, K, M = 4096, 4096, 8
    x = (torch.randn(M, K, device="cuda") * 0.5).to(torch.bfloat16)
    ws = [torch.randn(N, K, device="cuda") * 0.02 * (i + 1) for i in range(4)]
    quant = (lambda w: Q.quantize_4bit(w, blocksize=64, packed=True)) if bits == 4 else (lambda w: Q.quantize_8bit(w, blocksize=64))
    want = []
    for w in ws:
        q, s, z = quant(w)
        torch.cuda.synchronize()
        want.append(linear_wna16(x, q, s, z, None, bits=bits, blocksize=64, out_features=N).clone())
    torch.cuda.synchronize()
    bad = 0
    for rep in range(30):
        outs = []
        for w in ws:                                       # quantize -> GEMM -> quantize -> GEMM ..., back to back
            q, s, z = quant(w)
            outs.append(linear_wna16(x, q, s, z, None, bits=bits, blocksize=64, out_features=N))
        torch.cuda.synchronize()
        bad += sum(0 if torch.equal(a, b) else 1 for a, b in zip(outs, want))
    assert bad == 0
    # ... and behind a kernel of another library that writes them (a torch copy: it never releases dependents early,
    # so the GEMM grid starts only when the copy has completed)
    q, s, z = quant(ws[0])
    torch.cuda.synchronize()
    bad = 0
    for rep in range(30):
        q2, s2, z2 = torch.empty_like(q), torch.empty_like(s), torch.empty_like(z)
        q2.copy_(q); s2.copy_(s); z2.copy_(z)
        y = linear_wna16(x, q2, s2, z2, None, bits=bits, blocksize=64, out_features=N)
        q2.zero_()                                         # the next kernel on the stream overwrites the codes
        torch.cuda.synchronize()
        bad += 0 if torch.equal(y, want[0]) else 1
    assert bad == 0


def test_gemm_repeated_calls_leave_workspace_clean():
    """Stream-K counters are self-resetting: many calls on one workspace, identical results."""
    from quanta_b200.nn import linear_wna16
    N, K, M = 1024, 4096, 16
    w, x, b, q, s, z = make_case(N, K, M, 4, torch.bfloat16, seed=11)
    xd, bd = x.cuda(), b.cuda()
    y0 = linear_wna16(xd, q, s, z, bd, bits=4, blocksize=64, out_features=N)
    for _ in range(20):
        y = linear_wna16(xd, q, s, z, bd, bits=4, blocksize=64, out_features=N)
    assert torch.equal(y, y0)


def test_linear_modules_mirror_reference_api():
    from quanta_b200.nn import Linear4bit, Linear8bitLt
    torch.manual_seed(0)
    l4 = Linear4bit(512, 256, bias=True, compute_dtype=torch.bfloat16, quant_type="linear").cuda()
    l8 = Linear8bitLt(512, 256, bias=True, has_fp16_weights=False, threshold=6.0).cuda()
    assert l4.in_features == 512 and l4.out_features == 256 and l4.compute_dtype == torch.bfloat16
    assert l8.threshold == 6.0 and l8.has_fp16_weights is False
    for lin, dt in ((l4, torch.bfloat16), (l8, torch.float16)):
        w = lin.weight.detach().clone()
        x = torch.randn(3, 7, 512, device="cuda", dtype=dt)
        y = lin(x)
        assert y.shape == (3, 7, 256) and y.dtype == dt
        wd = lin.dequantize_weight(dt)
        ref = torch.nn.functional.linear(x.float(), wd.float(), lin.bias.float())
        assert float((y.float() - ref).abs().max() / ref.abs().max()) < TOL
        # and close to the unquantized layer (quantization error only)
        ref_fp = torch.nn.functional.linear(x.float(), w.float(), lin.bias.float())
        assert float((y.float() - ref_fp).abs().max() / ref_fp.abs().max()) < (0.15 if lin.bits == 4 else 0.02)
    with pytest.raises(NotImplementedError):
        Linear4bit(64, 64, quant_type="fp4").cuda()(torch.randn(1, 64, device="cuda", dtype=torch.float16))


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(128, 64, 1), (256, 512, 16), (384, 1024, 33), (1024, 4096, 64), (512, 2048, 256),
                                   (200, 320, 7)])
def test_nf4_gemm_matches_composition_oracle(dtype, shape):
    """F.linear(x, dequantize_4bit(idx, levels, absmax, "nf4").to(x.dtype)) in float64 (codes are bit-exact with
    the reference, tests/test_gpu_nf4.py)."""
    import quanta_b200 as Q
    from quanta_b200.nn import linear_nf4a16
    N, K, M = shape
    g = torch.Generator().manual_seed(N + K + M)
    w = torch.randn(N, K, generator=g) * 0.02
    x = torch.randn(M, K, generator=g).to(dtype)
    b = (torch.randn(N, generator=g) * 0.1).to(dtype)
    q, levels, am = Q.quantize_4bit(w.cuda(), quant_type="nf4", blocksize=64, packed=True)
    y = linear_nf4a16(x.cuda(), q, am, b.cuda(), blocksize=64, out_features=N)
    idx = O.unpack4(q.cpu().numpy())[: N * K].reshape(N, K)
    wd = O.dequantize_nf4(idx, am.cpu().numpy(), 64)
    wd = O._round_to(wd, "bf16" if dtype == torch.bfloat16 else "fp16")
    ref = x.float().numpy().astype(np.float64) @ wd.astype(np.float64).T + b.float().numpy().astype(np.float64)
    assert rel_err(y.float().cpu().numpy(), ref) < TOL


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("shape", [(128, 256, 1), (1000, 4096, 3), (136, 1536, 9), (264, 768, 5), (512, 11008, 2),
                                   (384, 2048, 16), (2048, 8192, 8)])
def test_nf4_small_batch_kernel(dtype, shape):
    """M <= 16, K % 256 == 0: NF4 goes through the weight-stream kernel as well (byte -> level-pair table in shared
    memory, csrc/gemm_small.cu).  Same oracle as above; the levels enter the MMA rounded to the activation type and the
    block's abs_max is applied in fp32, so the result is at least as close as the tcgen05 path's."""
    import quanta_b200 as Q
    from quanta_b200.nn import linear_nf4a16
    N, K, M = shape
    g = torch.Generator().manual_seed(7 * N + K + M)
    w = torch.randn(N, K, generator=g) * 0.02
    x = torch.randn(M, K, generator=g).to(dtype)
    b = (torch.randn(N, generator=g) * 0.1).to(dtype)
    q, levels, am = Q.quantize_4bit(w.cuda(), quant_type="nf4", blocksize=64, packed=True)
    xd, bd = x.cuda(), b.cuda()
    y = linear_nf4a16(xd, q, am, bd, blocksize=64, out_features=N)
    idx = O.unpack4(q.cpu().numpy())[: N * K].reshape(N, K)
    wd = O.dequantize_nf4(idx, am.cpu().numpy(), 64)
    ref = x.float().numpy().astype(np.float64) @ wd.astype(np.float64).T + b.float().numpy().astype(np.float64)
    err = rel_err(y.float().cpu().numpy(), ref)
    assert err < TOL, f"rel err {err:.3e} for {shape} {dtype}"
    for _ in range(3):                     # deterministic, counters left clean
        assert torch.equal(linear_nf4a16(xd, q, am, bd, blocksize=64, out_features=N), y)


def test_linear4bit_default_is_nf4():
    from quanta_b200.nn import Linear4bit
    torch.manual_seed(1)
    lin = Linear4bit(512, 256).cuda()                      # reference defaults: compute_dtype=float16, quant_type="nf4"
    w = lin.weight.detach().clone()
    x = torch.randn(5, 512, device="cuda", dtype=torch.float16)
    y = lin(x)
    assert y.shape == (5, 256) and y.dtype == torch.float16
    ref = torch.nn.functional.linear(x.float(), lin.dequantize_weight(torch.float16).float(), lin.bias.float())
    assert float((y.float() - ref).abs().max() / ref.abs().max()) < TOL
    ref_fp = torch.nn.functional.linear(x.float(), w.float(), lin.bias.float())
    assert float((y.float() - ref_fp).abs().max() / ref_fp.abs().max()) < 0.15


@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("M", [5, 48, 200])
@pytest.mark.parametrize("K", [512, 2048])
def test_scatter_epilogue_writes_every_output(bits, M, K):
    """Column-parallel entry: the tile is written at column col0 of each output buffer (pitch ldy)
    and nothing else in the buffers is touched."""
    import quanta_b200 as Q
    from quanta_b200.nn.functional import linear_wna16, linear_wna16_scatter
    N, ldy, col0 = 384, 1024, 256
    g = torch.Generator().manual_seed(M + bits)
    w = (torch.randn(N, K, generator=g) * 0.05).cuda()
    b = (torch.randn(N, generator=g) * 0.1).cuda().to(torch.bfloat16)
    x = torch.randn(M, K, generator=g).cuda().to(torch.bfloat16)
    qf = Q.quantize_4bit(w, blocksize=64, packed=True) if bits == 4 else Q.quantize_8bit(w, blocksize=64)
    ref = linear_wna16(x, *qf, b, bits=bits, blocksize=64, out_features=N)
    outs = [torch.full((M, ldy), 7.0, dtype=torch.bfloat16, device="cuda") for _ in range(3)]
    linear_wna16_scatter(x, *qf, b, ([o.data_ptr() for o in outs], ldy), col0, bits=bits, blocksize=64, out_features=N)
    torch.cuda.synchronize()
    for o in outs:
        assert torch.equal(o[:, col0:col0 + N], ref)
        assert bool((o[:, :col0] == 7.0).all()) and bool((o[:, col0 + N:] == 7.0).all())
