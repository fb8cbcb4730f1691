"""Comparison helpers shared by the CPU and GPU parity tests, and the inputs of the codebook (NF4 / nf8) oracle tests."""
import numpy as np
import pytest


def bits_equal(a, b):
    """Bit-exact equality of two float32 arrays (NaNs with equal payload match)."""
    a = np.ascontiguousarray(a, np.float32).reshape(-1)
    b = np.ascontiguousarray(b, np.float32).reshape(-1)
    return a.shape == b.shape and bool(np.array_equal(a.view(np.uint32), b.view(np.uint32)))


def assert_f32_bits(a, b, what="", zero_sign_free=False):
    """float32 arrays must match bit for bit.  ``zero_sign_free`` lets -0.0 match
    +0.0 (the reference's min() returns either, see oracle/oracle_np.py)."""
    a = np.ascontiguousarray(a, np.float32).reshape(-1)
    b = np.ascontiguousarray(b, np.float32).reshape(-1)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    ua, ub = a.view(np.uint32).copy(), b.view(np.uint32).copy()
    if zero_sign_free:
        ua[ua == 0x80000000] = 0
        ub[ub == 0x80000000] = 0
    # all NaNs compare equal (payload/sign of a produced NaN is not part of the contract)
    na, nb = np.isnan(a), np.isnan(b)
    assert np.array_equal(na, nb), f"{what}: NaN pattern differs"
    bad = (ua != ub) & ~na
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {a.size} float32 values differ; first at "
                           f"{int(np.argmax(bad))}: {a[np.argmax(bad)]!r} vs {b[np.argmax(bad)]!r}")


def assert_u8_equal(a, b, what=""):
    a = np.asarray(a).reshape(-1)
    b = np.asarray(b).reshape(-1)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    bad = a != b
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {a.size} codes differ; first at "
                           f"{int(np.argmax(bad))}: {a[np.argmax(bad)]} vs {b[np.argmax(bad)]}")


def ulp_diff(a, b):
    """Max distance in float32 ulps between two finite arrays."""
    a = np.ascontiguousarray(a, np.float32).reshape(-1)
    b = np.ascontiguousarray(b, np.float32).reshape(-1)

    def key(x):
        i = x.view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return int(np.max(np.abs(key(a) - key(b)))) if a.size else 0


# (shape, block, dtype, case) beyond each codebook oracle test's original four: 16-bit inputs, every block size from
# 16 to 512, inputs that take the per-tensor tail kernel (stored at a 1-element offset, so not 16-byte aligned; numel
# neither a multiple of 16 nor even), and abs-max values outside the hoisted-reciprocal window [2^-100, 2^100]: tiny,
# huge, zero, NaN and inf (see codebook_input)
CODEBOOK_EDGE_CASES = [pytest.param((512, 256), b, dt, None, id=f"{n}-{b}")
                       for n, dt in (("f16", "float16"), ("bf16", "bfloat16")) for b in (None, 64)] + \
                      [pytest.param((512, 256), b, "float32", None, id=f"block{b}") for b in (16, 32, 256, 512)] + [
    pytest.param((1000, 37), None, "float32", "offset", id="offset"),
    pytest.param((1000, 37), None, "bfloat16", "offset", id="offset-bf16"),
    pytest.param((333, 7), None, "float32", None, id="odd-numel"),
    pytest.param((512, 256), None, "float32", "tiny", id="tiny"),
    pytest.param((512, 256), 64, "float32", "tiny", id="tiny-64"),
    pytest.param((512, 256), None, "float32", "huge", id="huge"),
    pytest.param((512, 256), 64, "float32", "huge", id="huge-64"),
    pytest.param((512, 256), None, "float32", "zeros", id="zeros"),
    pytest.param((512, 256), None, "float32", "inf", id="inf"),
    pytest.param((512, 256), None, "float32", "specials", id="nan"),
    pytest.param((512, 256), 64, "float32", "specials", id="specials-64"),
]


def codebook_input(shape, dtype, case, seed):
    """Seeded ``randn * 0.02`` as a CUDA tensor of ``dtype``, and its float32 values for the oracle.
    case: None; "tiny" / "huge" (scaled by 1e-35 / 1e35); "zeros"; "inf" (one +inf); "specials" (flat elements 0-63
    zero, a NaN at 69, -inf at 137: with block 64 an all-zero block, a NaN block and an inf block); "offset" (stored
    one element into its buffer)."""
    import torch
    dtype = getattr(torch, dtype) if isinstance(dtype, str) else dtype
    x = torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * 0.02
    flat = x.view(-1)
    if case == "tiny":
        x *= 1e-35
    elif case == "huge":
        x *= 1e35
    elif case == "zeros":
        x.zero_()
    elif case == "inf":
        flat[100] = float("inf")
    elif case == "specials":
        flat[:64] = 0.0
        flat[69] = float("nan")
        flat[137] = -float("inf")
    x = x.to(dtype)
    xf = x.float().numpy()
    if case == "offset":
        buf = torch.empty(x.numel() + 1, dtype=dtype, device="cuda")
        buf[1:].copy_(x.reshape(-1))
        return buf[1:].view(shape), xf
    return x.cuda(), xf
