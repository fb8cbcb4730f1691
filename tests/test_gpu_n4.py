"""GPU parity tests of nf8 / fp4 / fp8 (row N4) against golden vectors produced by the unmodified reference
(tests/golden/make_tables_n4.py) and against the numpy oracle: codes, abs_max and dequantized values bit-exact."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import CODEBOOK_EDGE_CASES, codebook_input
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu
Z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "quanta_golden_n4.npz"))
MANIFEST = json.loads(str(Z["manifest"]))


def same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def test_fp4_fp8_match_reference_golden():
    import quanta_b200 as Q
    for c in MANIFEST:
        if c["kind"] not in ("fp4", "fp8"):
            continue
        x = torch.from_numpy(Z[f"{c['name']}/x"]).cuda()
        if c["kind"] == "fp4":
            q, none, bias = Q.quantize_4bit(x, quant_type="fp4")
            d = Q.dequantize_4bit(q, None, bias, quant_type="fp4")
        else:
            q, none, bias = Q.quantize_8bit(x, quant_type="fp8")
            d = Q.dequantize_8bit(q, None, bias, quant_type="fp8")
        assert none is None and bias == (1 if c["kind"] == "fp4" else 7)
        assert q.dtype == torch.uint8 and q.shape == x.shape
        assert np.array_equal(q.cpu().numpy(), Z[f"{c['name']}/q"]), c
        assert same_bits(d.cpu().numpy(), Z[f"{c['name']}/deq"]), c


def test_nf8_matches_reference_golden():
    import quanta_b200 as Q
    lv_ref = O.nf8_levels()
    for c in MANIFEST:
        if c["kind"] != "nf8":
            continue
        x = torch.from_numpy(Z[f"{c['name']}/x"]).cuda()
        idx, levels, am = Q.quantize_8bit(x, quant_type="nf8")
        assert np.array_equal(levels.cpu().numpy().view(np.uint32), lv_ref.view(np.uint32))
        assert np.array_equal(idx.cpu().numpy(), Z[f"{c['name']}/q"]), c
        assert same_bits(am.cpu().numpy(), Z[f"{c['name']}/absmax"]), c
        d = Q.dequantize_8bit(idx, levels, am, quant_type="nf8")
        assert same_bits(d.cpu().numpy(), Z[f"{c['name']}/deq"]), c


@pytest.mark.parametrize("shape,block,dtype,case", [
    pytest.param(shape, block, "float32", None, id=f"shape{i}-{block}")
    for i, (shape, block) in enumerate([((2048, 1024), None), ((2048, 1024), 64), ((1000, 37), None), ((512, 256), 128)])
] + CODEBOOK_EDGE_CASES)
def test_nf8_large_random_matches_oracle(shape, block, dtype, case):
    import quanta_b200 as Q
    x, xf = codebook_input(shape, dtype, case, seed=9)
    idx, levels, am = Q.quantize_8bit(x, quant_type="nf8", blocksize=block)
    io, ao = O.quantize_nf8(xf, block)
    assert np.array_equal(idx.cpu().numpy(), io)
    assert same_bits(am.cpu().numpy(), ao)
    d = Q.dequantize_8bit(idx, levels, am, quant_type="nf8", blocksize=block)
    assert same_bits(d.cpu().numpy(), O.dequantize_nf8(io, ao, block))


@pytest.mark.parametrize("bits", [4, 8])
@pytest.mark.parametrize("scale", [1.0, 0.02, 300.0])
def test_fp_large_random_matches_oracle(bits, scale):
    import quanta_b200 as Q
    g = torch.Generator().manual_seed(bits)
    x = torch.randn(1537, 1031, generator=g) * scale
    x[0, :8] = torch.tensor([0.0, -0.0, 1e-40, -1e-40, 3e38, -3e38, float("inf"), -float("inf")])
    fn, dq, qt = (Q.quantize_4bit, Q.dequantize_4bit, "fp4") if bits == 4 else (Q.quantize_8bit, Q.dequantize_8bit, "fp8")
    q, _, bias = fn(x.cuda(), quant_type=qt)
    qo = O.quantize_fp(x.numpy(), bits)
    assert np.array_equal(q.cpu().numpy(), qo)
    assert same_bits(dq(q, None, bias, quant_type=qt).cpu().numpy(), O.dequantize_fp(qo, bits, bias))
    # every code decodes like the reference formula, in the half-precision output types too
    codes = torch.arange(256 if bits == 8 else 16, dtype=torch.uint8).cuda()
    want = O.dequantize_fp(codes.cpu().numpy(), bits, bias)
    for od in (torch.float32, torch.bfloat16, torch.float16):
        got = dq(codes, None, bias, quant_type=qt, out_dtype=od)
        assert torch.equal(got.cpu(), torch.from_numpy(want).to(od))


def test_fp_exponent_thresholds_exhaustive_neighbourhood():
    """+-64 floats around every derived exponent threshold, both signs: the field changes exactly there."""
    import quanta_b200 as Q
    t = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "quanta_tables_n4.npz"))
    for bits, key in ((4, "fp4_exp_thresholds"), (8, "fp8_exp_thresholds")):
        thr = t[key].astype(np.float32)
        bitsv = thr.view(np.uint32).astype(np.int64)[:, None] + np.arange(-64, 65)[None, :]
        x = bitsv.astype(np.uint32).view(np.float32).reshape(-1)
        x = np.concatenate([x, -x])
        fn, qt = (Q.quantize_4bit, "fp4") if bits == 4 else (Q.quantize_8bit, "fp8")
        q = fn(torch.from_numpy(x).cuda(), quant_type=qt)[0].cpu().numpy()
        assert np.array_equal(q, O.quantize_fp(x, bits))
