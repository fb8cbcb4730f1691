"""The batched blockwise quantize stream (quanta_quantize_block_batch): several multi-tensor launches per call that
overlap (each releases the next one early; the next waits for it before it exits), and per-tensor fallbacks in the
middle of a batch.  Every result must equal one quantize_4bit call per tensor bit for bit.  Work queued right after
the call reads outputs of its FIRST launch, eagerly and inside a CUDA graph, and must see them finished.  That part can
only catch a broken chain by chance: the first launch nearly always completes long before the last one exits, so it
does not prove the ordering (the argument for it is in common.cuh, next to pdl_wait)."""
import numpy as np
import pytest
import torch

from helpers import assert_f32_bits, assert_u8_equal
from oracle import oracle_np as O

pytestmark = pytest.mark.gpu

# 40 tensors = 3 launches of at most 16 (4 when tensor FALLBACK breaks the second one).  Tiles are 256 rows of 32
# elements (8192 elements); 2 CTAs per SM are resident.  The shapes give tensors with one partial tile, with fewer
# tiles than the resident CTAs, with a tile count that is not a multiple of them and with several tiles per CTA; the
# last launch has fewer tiles than there are resident CTAs.
BIG = [(1024, 2048), (4096, 4096), (64, 64), (1000, 192), (11008, 512), (512, 1024), (2368, 1024), (3, 4096)]
SMALL = [(64, 64), (1000, 192), (512, 1024), (3, 4096), (128, 320), (256, 256), (7, 64), (512, 512)]
SHAPES = BIG * 4 + SMALL
FALLBACK = 20          # as a view at a 4-byte offset it is not 16-byte aligned and takes the per-tensor generic kernel


@pytest.fixture(scope="module")
def Q():
    import quanta_b200
    assert torch.cuda.is_available()
    g = torch.Generator(device="cuda").manual_seed(5)
    ACT["x"] = torch.randn(8, SHAPES[0][1], generator=g, device="cuda").to(torch.bfloat16)   # not created in a capture
    return quanta_b200


def make_inputs(dtype, fallback):
    g = torch.Generator(device="cuda").manual_seed(77)
    ts = []
    for i, (r, c) in enumerate(SHAPES):
        x = (torch.randn(r * c + 2, generator=g, device="cuda") * (0.02 * (i + 1))).to(dtype)
        off = 4 // x.element_size() if fallback and i == FALLBACK else 0
        t = x[off:off + r * c].view(r, c)
        assert (t.data_ptr() % 16 != 0) == (off != 0)
        ts.append(t)
    return ts


def per_tensor(Q, ts):
    ref = [Q.quantize_4bit(t, blocksize=64, packed=True) for t in ts]
    torch.cuda.synchronize()
    return [tuple(a.clone() for a in r) for r in ref]


def check_equal(got, ref, what):
    for i, ((q, s, z), (rq, rs, rz)) in enumerate(zip(got, ref)):
        w = f"{what} tensor {i} {SHAPES[i]}"
        assert_u8_equal(q.cpu().numpy(), rq.cpu().numpy(), w + " codes")
        assert_f32_bits(s.cpu().numpy(), rs.cpu().numpy(), w + " scale")
        assert_f32_bits(z.cpu().numpy(), rz.cpu().numpy(), w + " zp")


ACT = {}


def downstream(Q, outs):
    """Work queued right behind the call, reading outputs of its first launch: a batched dequantize of the first
    16 tensors and a W4A16 linear on tensor 0 (1024 x 2048)."""
    from quanta_b200.nn import linear_wna16
    first = list(range(16))
    deq = Q.dequantize_4bit_many([outs[i][0] for i in first], [outs[i][1] for i in first], [outs[i][2] for i in first],
                                 blocksize=64, packed=True, shapes=[SHAPES[i] for i in first])
    x = ACT["x"]
    y = linear_wna16(x, outs[0][0], outs[0][1], outs[0][2], None, bits=4, blocksize=64, out_features=SHAPES[0][0])
    return deq, y


def check_downstream(Q, got, ref_outs, what):
    deq, y = got
    rdeq, ry = downstream(Q, ref_outs)
    torch.cuda.synchronize()
    for i, (a, b) in enumerate(zip(deq, rdeq)):
        assert_f32_bits(a.cpu().numpy(), b.cpu().numpy(), f"{what}: dequantize of tensor {i}")
    ya, yb = y.float().cpu().numpy(), ry.float().cpu().numpy()
    err = np.abs(ya - yb).max() / (np.abs(yb).max() + 1e-30)
    assert err < 1e-3, f"{what}: linear_wna16 on tensor 0 differs, rel err {err:.3e}"


@pytest.mark.parametrize("fallback", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_many_equals_per_tensor_eager(Q, dtype, fallback):
    ts = make_inputs(dtype, fallback)
    ref = per_tensor(Q, ts)
    for rep in range(2):
        outs = Q.quantize_4bit_many(ts, blocksize=64, packed=True)
        got = downstream(Q, outs)               # no synchronisation between the call and its readers
        torch.cuda.synchronize()
        check_equal(outs, ref, f"eager rep {rep}")
        check_downstream(Q, got, ref, f"eager rep {rep}")


@pytest.mark.parametrize("fallback", [False, True])
def test_many_equals_per_tensor_graph(Q, fallback):
    ts = make_inputs(torch.float32, fallback)
    ref = per_tensor(Q, ts)
    Q.quantize_4bit_many(ts, blocksize=64, packed=True)        # warm-up outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = Q.quantize_4bit_many(ts, blocksize=64, packed=True)
        got = downstream(Q, outs)
    for rep in range(3):
        for o in outs:
            for a in o:
                a.fill_(0)
        graph.replay()
        torch.cuda.synchronize()
        check_equal(outs, ref, f"graph replay {rep}")
        check_downstream(Q, got, ref, f"graph replay {rep}")


def test_many_matches_oracle_on_small_tensors(Q):
    """The per-tensor reference above runs the single-tensor stream, which shares the schedule: anchor both to the
    oracle on the tensors that are cheap to check on the host, the unaligned fallback included."""
    ts = make_inputs(torch.float32, True)
    outs = Q.quantize_4bit_many(ts, blocksize=64, packed=True)
    torch.cuda.synchronize()
    for i, t in enumerate(ts):
        if t.numel() > 1 << 20:
            continue
        po, so, zo = O.quantize4_block_pack(t.cpu().numpy(), 64)
        w = f"tensor {i} {SHAPES[i]}"
        assert_u8_equal(outs[i][0].cpu().numpy(), po, w + " codes")
        assert_f32_bits(outs[i][1].cpu().numpy(), so, w + " scale")
        assert_f32_bits(outs[i][2].cpu().numpy(), zo, w + " zp", zero_sign_free=True)


def test_input_error_after_a_release_still_completes_the_chain(Q):
    """Through the C ABI (the Python API rejects the bad size first): tensor 18 has a size that is not a multiple of
    the block, so the call fails after the first launch has released the second.  The pending group (tensors 16 and
    17) is still launched, the call returns QUANTA_EINVAL, and tensors 0-17 are quantized."""
    import ctypes as C
    from quanta_b200 import _host, _lib
    ts = make_inputs(torch.float32, False)[:20]
    ref = per_tensor(Q, ts)
    outs = [(torch.empty(t.numel() // 2, dtype=torch.uint8, device="cuda"),
             torch.empty(t.numel() // 64, dtype=torch.float32, device="cuda"),
             torch.empty(t.numel() // 64, dtype=torch.float32, device="cuda")) for t in ts]
    numels = [t.numel() for t in ts]
    numels[18] = 65
    k = len(ts)
    arr = C.c_void_p * k
    st = _lib.lib().quanta_quantize_block_batch(
        arr(*[t.data_ptr() for t in ts]), (C.c_int64 * k)(*numels), k, _host.dtype_code(ts[0]), 64, 4, 1,
        arr(*[o[0].data_ptr() for o in outs]), arr(*[o[1].data_ptr() for o in outs]), arr(*[o[2].data_ptr() for o in outs]),
        _host.stream_ptr(torch.device("cuda", torch.cuda.current_device())))
    assert st == -1                                        # QUANTA_EINVAL
    torch.cuda.synchronize()
    check_equal(outs[:18], ref[:18], "before the bad tensor")
