"""GPU parity tests of the NF4 codebook path (row N1) against golden vectors produced by the
unmodified reference and against the numpy oracle: codes and abs_max bit-exact, dequantized
values bit-exact."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import CODEBOOK_EDGE_CASES, codebook_input
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu
Z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "quanta_golden_nf4.npz"))
MANIFEST = json.loads(bytes(Z["manifest"]).decode())


def same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def test_nf4_matches_reference_golden():
    import quanta_b200 as Q
    for c in MANIFEST:
        x = torch.from_numpy(Z[f"{c['name']}/x"]).cuda()
        idx, levels, am = Q.quantize_4bit(x, quant_type="nf4", blocksize=c["block"])
        assert idx.dtype == torch.uint8 and idx.shape == x.shape
        assert np.array_equal(idx.cpu().numpy(), Z[f"{c['name']}/idx"]), c
        assert same_bits(am.cpu().numpy(), Z[f"{c['name']}/absmax"]), c
        assert np.array_equal(levels.cpu().numpy().view(np.uint32), Z["levels"].view(np.uint32))
        d = Q.dequantize_4bit(idx, levels, am, quant_type="nf4", blocksize=c["block"])
        assert same_bits(d.cpu().numpy(), Z[f"{c['name']}/deq"]), c


@pytest.mark.parametrize("shape,block,dtype,case", [
    pytest.param(shape, block, "float32", None, id=f"shape{i}-{block}")
    for i, (shape, block) in enumerate([((4096, 1024), None), ((4096, 1024), 64), ((1000, 37), None), ((512, 256), 128)])
] + CODEBOOK_EDGE_CASES)
@pytest.mark.parametrize("packed", [False, True])
def test_nf4_large_random_matches_oracle(shape, block, dtype, case, packed):
    import quanta_b200 as Q
    x, xf = codebook_input(shape, dtype, case, seed=5)
    idx, levels, am = Q.quantize_4bit(x, quant_type="nf4", blocksize=block, packed=packed)
    io, ao = O.quantize_nf4(xf, block)
    got = idx.cpu().numpy()
    if packed:
        got = O.unpack4(got)[: xf.size].reshape(shape)
    assert np.array_equal(got, io)
    assert same_bits(am.cpu().numpy(), ao)
    d = Q.dequantize_4bit(idx, levels, am, quant_type="nf4", blocksize=block, packed=packed, shape=shape)
    assert same_bits(d.cpu().numpy(), O.dequantize_nf4(io, ao, block))
    if np.isfinite(xf).all():
        # size-independent property: every value lands on one of the 16 levels times its abs_max, error <= half a gap
        assert float(np.abs(d.cpu().numpy() - xf).max()) <= 0.16 * float(np.abs(xf).max())


@pytest.mark.parametrize("packed", [True, False])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_nf4_many_equals_one_call_per_tensor(packed, dtype):
    """The batched launch (and the TMA-stream path behind blocksize=64) give the bits of the per-tensor calls,
    which the tests above pin to the reference."""
    import quanta_b200 as Q
    g = torch.Generator().manual_seed(11)
    shapes = [(256, 512), (300, 64), (1, 64), (1024, 1024), (77, 128), (4096, 320)]
    xs = [(torch.randn(*sh, generator=g) * (0.02 + i)).to(dtype).cuda() for i, sh in enumerate(shapes)]
    xs[2].zero_()                                     # an all-zero block: 0/0 -> code 0
    many = Q.quantize_nf4_many(xs, blocksize=64, packed=packed)
    for x, (q, lv, am) in zip(xs, many):
        io, ao = O.quantize_nf4(x.float().cpu().numpy().reshape(-1), 64)
        got = q.cpu().numpy().reshape(-1)
        if packed:
            got = O.unpack4(got)[: x.numel()]
        assert np.array_equal(got, io)
        assert same_bits(am.cpu().numpy(), ao)
        q1, _, am1 = Q.quantize_4bit(x, quant_type="nf4", blocksize=64, packed=packed)
        assert torch.equal(q1.reshape(-1), q.reshape(-1)) and torch.equal(am1, am)
