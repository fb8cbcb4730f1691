#!/usr/bin/env python
"""bench.py — headline benchmark of the weight-quantization hot path.

N = 1 (BASELINE.json configs[1]): 4-bit blockwise (blocksize 64) quantize + nibble-pack of all
Llama-2-7B-shaped decoder linears (32 x {4x[4096,4096], 2x[11008,4096], [4096,11008]} = 6.476 G fp32
elements, 25.9 GB) on one B200.  A "step" is one pass over all 224 matrices.

  value     algorithmic GB/s (4.625 B/elem: 4 read + 0.5 packed + 8/64 scale+zp), inputs resident in
            HBM, the step's launches replayed as one CUDA graph, timed with CUDA events
  e2e       the same metric through the public API with HOST buffers: pinned host -> device copies of
            every matrix and device -> host copies of every result inside the timed region
  roofline  achieved GB/s of the dominant kernel against the measured HBM peak in MEASURED_PEAKS.json;
            `traffic` is read from the committed ncu capture of that kernel (profiles/*.json)
  cpu_baseline  the UNMODIFIED reference (oracle/_ref, vendored by `make -C oracle`) on the host cores,
            bounded sample; the C/OpenMP port of the same arithmetic next to it (`c_port_value`)
  secondary the other half of BASELINE.json's metric, measured in the same run: W4A16 / W8A16 / NF4
            dequant-GEMM on the Llama-3-8B shapes (config 3), dequantize, the config-1 round trip

N > 1 (configs[4], launched by torchrun): 16 Llama-3-70B-shaped decoder layers (13.69 G elements, 54.8 GB
fp32 — FIXED total work, strong scaling) row-sharded over the ranks: every rank quantizes rows
row_shard(out, N, rank, 128) of every matrix with no data-path collective; then the tensor-parallel
dequant-GEMM (local kernel, NCCL all-gather, gather fused into the GEMM epilogue over NVLink) is timed
and checked in `secondary.tp`.

`--impl reference` times the reference's own CPU implementation of the path on the host cores: the
unmodified package from oracle/_ref (kind "reference"; oracle/oracle_torch.py, kind "port", only if the
vendored copy is missing).

`--dump-outputs DIR` writes a fixed, seeded sample of what the timed step returned in its last replay to
DIR/packed.npy, DIR/scale.npy and DIR/zero_point.npy (float32, under 64 MB in all), so that two builds run
with the same arguments can be compared output for output.
"""
import argparse
import glob
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree, which may be read-only

LLAMA2_7B_LAYER = [(4096, 4096)] * 4 + [(11008, 4096)] * 2 + [(4096, 11008)]
LLAMA3_70B_LAYER = [(8192, 8192)] * 2 + [(1024, 8192)] * 2 + [(28672, 8192)] * 2 + [(8192, 28672)]
N_LAYERS = 32
N_LAYERS_70B = 16                       # of 80: fixed total work of the N > 1 runs (54.8 GB fp32)
BYTES_PER_ELEM = 4.0 + 0.5 + 8.0 / 64.0
BLOCK = 64
METRIC = "quantize/dequantize GB/s vs HBM peak (4-bit block-64 quantize+pack, algorithmic bytes)"
WORKLOAD = "llama2-7b decoder linears, fp32 -> 4-bit block-64 quantize+pack"
WORKLOAD_70B = ("llama3-70b decoder linears (%d of 80 layers), row-sharded over the ranks, fp32 -> 4-bit block-64 "
                "quantize+pack" % N_LAYERS_70B)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
        return {"hbm": float(pk["hbm_gbs"]), "tf": float(pk["bf16_tflops"]), "tf_sustained": float(pk["bf16_tflops_sustained"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    except Exception:
        return {"hbm": 6650.0, "tf": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(kernel_substr):
    """DRAM bytes per launch of the dominant kernel from the newest committed ncu summary (profiles/*traffic*.json,
    written by tools/ncu_summary.py from an `ncu --set full` capture)."""
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "*traffic*.json"))):
        try:
            for rec in json.load(open(path)):
                if kernel_substr in rec.get("kernel", ""):
                    best = dict(rec, file=os.path.relpath(path, ROOT))
        except Exception:
            continue
    return best


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons with NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path
# ---------------------------------------------------------------------------------------------

def cpu_sample():
    """One decoder layer (7 matrices, 202 M elements) of synthetic weights for the CPU arm."""
    import numpy as np
    rng = np.random.default_rng(1234)
    return [rng.standard_normal(r * c, dtype=np.float32) * np.float32(0.02) for r, c in LLAMA2_7B_LAYER]


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def reference_impl():
    """(quantize4_block_pack(tensor, block) -> (packed, scale, zp), kind, description).  The unmodified reference
    package when oracle/_ref holds it: blockwise-B is its per_channel branch on x.reshape(-1, B).t()
    (Quanta/functional/quantization.py:77-84, SURVEY A.1), packing is Quanta/utils/utils.py:23-35."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if os.path.isdir(os.path.join(ref_dir, "Quanta")):
        sys.path.insert(0, ref_dir)
        try:
            from Quanta.functional.quantization import quantize_4bit
            from Quanta.utils.utils import pack_4bit_tensor
        finally:
            sys.path.pop(0)

        def run(t, block):
            q, scale, zp = quantize_4bit(t.reshape(-1, block).t(), "linear", True)
            packed, _ = pack_4bit_tensor(q.t().contiguous())
            return packed, scale, zp
        return run, "reference", "unmodified reference (oracle/_ref/Quanta: quantize_4bit per_channel on x.reshape(-1,64).t() + pack_4bit_tensor)"
    from oracle import oracle_torch as OT
    return (lambda t, block: OT.quantize4_block_pack(t, block)), "port", "oracle/oracle_torch.py (oracle/_ref not built)"


def time_cpu_reference(mats, layers_per_step, reps, warmup):
    import torch
    run, kind, what = reference_impl()
    threads = host_threads()
    torch.set_num_threads(threads)
    ts = [torch.from_numpy(m).reshape(r, c) for m, (r, c) in zip(mats, LLAMA2_7B_LAYER)]
    elems = sum(t.numel() for t in ts) * layers_per_step
    times = []
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        for _ in range(layers_per_step):
            for t in ts:
                run(t, BLOCK)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return elems, times, torch.get_num_threads(), kind, what


def time_cpu_c_port(mats, reps, warmup):
    """C/OpenMP port of the arithmetic (oracle/quanta_oracle.c), as built by build()."""
    from oracle import oracle_c as OC
    elems = sum(m.size for m in mats)
    times = []
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        for m in mats:
            OC.quantize4_block_pack(m, BLOCK)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return elems, times, OC.num_threads()


def run_reference(args, rank):
    """CPU arm (rank 0 only): the reference's implementation on all host threads, same metric and config."""
    if rank != 0:
        return
    mats = cpu_sample()
    # size the step so that the whole run ends within a few minutes: time one layer, then take as many of
    # the 32 layers per step as fit a ~150 s budget
    _, t1, _, _, _ = time_cpu_reference(mats, 1, 1, 1)
    total_steps = args.steps + args.warmup
    layers = int(max(1, min(N_LAYERS, 150.0 / max(total_steps, 1) / max(t1[0], 1e-3))))
    elems, times, threads, kind, what = time_cpu_reference(mats, layers, args.steps, args.warmup)
    t = sum(times) / len(times)
    value = elems * BYTES_PER_ELEM / t / 1e9
    same = layers == N_LAYERS
    sample = ("%d of 32 decoder layers per step (%d matrices, %d elements; the layer's 7 random matrices are revisited); "
              "%s; %d intra-op threads" % (layers, 7 * layers, elems, what, threads))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "blocksize": BLOCK, "sample": sample, "same_config": same},
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------

def graph_time_us(fn, reps, torch):
    """Device time per call of fn(i), i = 0..reps-1, replayed from one CUDA graph (CUDA events)."""
    for i in range(3):
        fn(i)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn(0)                                   # per-stream workspaces exist before capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        outs = [fn(i) for i in range(reps)]
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    del g, outs
    return us


def secondary_single_gpu(device, pk, torch, Q):
    """The rest of BASELINE.json's metric on one GPU: config 3 (dequant-GEMM TFLOP/s on the Llama-3-8B
    shapes), dequantize GB/s, config 1 (8-bit round trip of a 4096 x 4096 fp32 weight).  Every number is
    device time under CUDA-graph replay over rotating inputs whose footprint exceeds L2."""
    from quanta_b200.nn import linear_wna16, linear_nf4a16
    HBM, TF, TFS = pk["hbm"], pk["tf"], pk["tf_sustained"]
    out = {"note": "CUDA-graph replay, rotating copies > L2, CUDA events; frac = binding-roof time / measured time "
                   "(HBM roof: algorithmic bytes / hbm_gbs; tensor roof: flops / BURST bf16 peak)", "gemm": [], "streams": []}
    launches = 0
    reps = 24
    for (N, K) in ((4096, 14336), (14336, 4096)):
        for fmt in ("W4A16", "W8A16", "NF4A16"):
            nf4 = fmt == "NF4A16"
            bits = 8 if fmt == "W8A16" else 4
            wbytes = N * K * bits // 8 + (N * K // 64) * (4 if nf4 else 8)
            copies = max(4, int(300e6 // wbytes) + 1)
            ws = []
            for i in range(copies):
                w = torch.empty(N, K, device=device).normal_(0.0, 0.02)
                if nf4:
                    q_, _, am_ = Q.quantize_4bit(w, quant_type="nf4", blocksize=64, packed=True)
                    ws.append((q_, am_))
                else:
                    ws.append(Q.quantize_4bit(w, blocksize=64, packed=True) if bits == 4 else Q.quantize_8bit(w, blocksize=64))
                del w
            for M in (1, 16, 64, 128, 256):
                x = torch.randn(M, K, device=device).to(torch.bfloat16)
                if nf4:
                    fn = lambda i: linear_nf4a16(x, *ws[i % copies], None, blocksize=64, out_features=N)
                else:
                    fn = lambda i: linear_wna16(x, *ws[i % copies], None, bits=bits, blocksize=64, out_features=N)
                us = graph_time_us(fn, reps, torch)
                launches += reps
                flops = 2.0 * M * N * K
                abytes = wbytes + 2 * M * K + 2 * M * N
                t_hbm, t_tc = abytes / HBM / 1e3, flops / TF / 1e6          # microseconds
                bound = "hbm" if t_hbm >= t_tc else "tensor"
                out["gemm"].append({"op": fmt, "N": N, "K": K, "M": M, "us": round(us, 2), "TFLOPs": round(flops / us / 1e6, 1),
                                    "GBps": round(abytes / us / 1e3, 1), "bound": bound,
                                    "frac": round(max(t_hbm, t_tc) / us, 3),
                                    "frac_sustained_peak": round(max(t_hbm, flops / TFS / 1e6) / us, 3)})
            del ws
            torch.cuda.empty_cache()

    def stream_case(name, shape, alg_bytes, make, fn, copies, reps=20):
        nonlocal launches
        ins = [make(i) for i in range(copies)]
        us = graph_time_us(lambda i: fn(ins[i % copies]), reps, torch)
        launches += reps
        gbs = alg_bytes / us / 1e3
        out["streams"].append({"op": name, "shape": list(shape), "alg_bytes": alg_bytes, "us": round(us, 2),
                               "GBps": round(gbs, 1), "frac": round(gbs / HBM, 3)})
        del ins
        torch.cuda.empty_cache()

    def randn(shape, i, scale=0.02):
        g = torch.Generator(device=device).manual_seed(100 + i)
        return torch.randn(shape, device=device, generator=g) * scale

    for shape in ((4096, 4096), (11008, 4096)):
        n = shape[0] * shape[1]
        copies = max(3, int(400e6 // (n * 4)) + 1)
        stream_case("quantize_8bit per-tensor (config 1, A1)", shape, n * 5.0, lambda i: randn(shape, i, 1.0),
                    lambda t: Q.quantize_8bit(t), copies)
        stream_case("dequantize_8bit per-tensor (config 1, A4)", shape, n * 5.0, lambda i: Q.quantize_8bit(randn(shape, i, 1.0)),
                    lambda t: Q.dequantize_8bit(*t), copies)
        stream_case("quantize_8bit + dequantize_8bit round trip (config 1)", shape, n * 10.0, lambda i: randn(shape, i, 1.0),
                    lambda t: Q.dequantize_8bit(*Q.quantize_8bit(t)), copies)
        stream_case("quantize_4bit block-64 + pack, one matrix (A3+P1)", shape, n * 4.625, lambda i: randn(shape, i),
                    lambda t: Q.quantize_4bit(t, blocksize=64, packed=True), copies)
        stream_case("dequantize_4bit packed block-64 -> fp32 (P2+A4)", shape, n * 4.625,
                    lambda i: Q.quantize_4bit(randn(shape, i), blocksize=64, packed=True),
                    lambda t: Q.dequantize_4bit(*t, blocksize=64, packed=True, shape=shape), copies)
        stream_case("quantize_8bit per_channel dim 0 (A3)", shape, n * 5.0, lambda i: randn(shape, i, 1.0),
                    lambda t: Q.quantize_8bit(t, per_channel=True), copies)

        def codes(i):
            g = torch.Generator(device=device).manual_seed(i)
            return torch.randint(0, 16, (n,), device=device, dtype=torch.uint8, generator=g)
        stream_case("pack_4bit_tensor (P1)", shape, n * 1.5, codes, lambda c: Q.pack_4bit_tensor(c), max(copies, 12))

    # config 4: LLM.int8()-style outlier split on OPT-6.7B shapes against an int8 tensor peak measured here (cuBLASLt)
    try:
        from quanta_b200.nn import int8_outlier_matmul, rowwise_quantize_sym
        a8 = torch.randint(-127, 127, (8192, 8192), device=device, dtype=torch.int8)
        b8 = torch.randint(-127, 127, (8192, 8192), device=device, dtype=torch.int8).t()
        for _ in range(3):
            torch._int_mm(a8, b8)
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a8, b8); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        int8_peak = 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12
        del a8, b8
        out["outlier"] = [{"int8_tensor_peak_TOPs": round(int8_peak, 1), "how": "torch._int_mm (cuBLASLt int8) 8192^3, best of 6"}]
        cols = [7, 513, 1024, 2049, 3071, 4000]
        for (N, K) in ((4096, 4096), (16384, 4096), (4096, 16384)):
            copies = max(3, int(300e6 // (N * K)) + 1)
            wq = [rowwise_quantize_sym(torch.empty(N, K, device=device).normal_(0.0, 0.02)) for _ in range(copies)]
            for M in (1, 16, 256, 2048):
                x = torch.randn(M, K, device=device)
                x[:, cols] *= 20.0
                x = x.to(torch.bfloat16)
                us = graph_time_us(lambda i: int8_outlier_matmul(x, wq[i % copies][0], wq[i % copies][1], threshold=6.0), 12, torch)
                launches += 12 * 4
                flops = 2.0 * M * N * K
                nbytes = N * K + 4 * N + 2 * M * K + 2 * M * N
                t_hbm, t_tc = nbytes / HBM / 1e3, flops / int8_peak / 1e6
                out["outlier"].append({"op": "int8_outlier_matmul", "N": N, "K": K, "M": M, "us": round(us, 2),
                                       "TOPs": round(flops / us / 1e6, 1), "bound": "hbm" if t_hbm >= t_tc else "tensor(int8)",
                                       "frac": round(max(t_hbm, t_tc) / us, 3)})
            del wq
            torch.cuda.empty_cache()
    except Exception as ex:                                  # noqa: BLE001 - the contract line must not depend on this row
        out["outlier"] = [{"skipped": "%s: %s" % (type(ex).__name__, ex)}]

    # the blockwise dequantize as ONE launch over a decoder layer's 7 matrices (quanta_dequantize_block_batch)
    layer = [(4096, 4096)] * 4 + [(11008, 4096)] * 2 + [(4096, 11008)]
    elems = sum(a * b for (a, b) in layer)

    def layer_codes(i):
        ws = [randn(sh, 10 * i + j) for j, sh in enumerate(layer)]
        qs = Q.quantize_4bit_many(ws, blocksize=BLOCK, packed=True)
        return [t[0] for t in qs], [t[1] for t in qs], [t[2] for t in qs]
    stream_case("dequantize_4bit_many packed block-64 -> fp32: one decoder layer, 7 matrices, 1 launch", (elems,), elems * 4.625,
                layer_codes, lambda t: Q.dequantize_4bit_many(t[0], t[1], t[2], blocksize=BLOCK, packed=True, shapes=layer), 3, reps=6)
    return out, launches


DUMP_BYTES = 60_000_000                 # --dump-outputs: all files of all ranks together
DUMP_NAMES = ("packed", "scale", "zero_point")


def dump_outputs(out_dir, outs, rank, world, torch):
    """Write a sample of one step's results: for each of the three arrays quantize_4bit returns, the values at
    seeded random positions (drawn with replacement, sorted) of all matrices' arrays laid end to end in step
    order, as float32 (packed bytes as their integer values).  The positions depend only on the array sizes,
    so runs with the same arguments sample the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = DUMP_BYTES // 4 // len(DUMP_NAMES) // world
    prefix = "rank%d_" % rank if world > 1 else ""
    for k, name in enumerate(DUMP_NAMES):
        parts = [o[k].reshape(-1) for o in outs]
        ends = torch.tensor([p.numel() for p in parts]).cumsum(0)
        total = int(ends[-1])
        if total <= n:
            idx = torch.arange(total)
        else:
            idx = torch.randint(0, total, (n,), generator=torch.Generator().manual_seed(1000 + k)).sort().values
        cuts = torch.searchsorted(idx, ends).tolist()
        vals, lo, start = [], 0, 0
        for p, hi, end in zip(parts, cuts, ends.tolist()):
            if hi > lo:
                vals.append(p[(idx[lo:hi] - start).to(p.device)].float().cpu())
            lo, start = hi, end
        np.save(os.path.join(out_dir, prefix + name + ".npy"), torch.cat(vals).numpy())


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import quanta_b200 as Q
    from quanta_b200.sharding import row_shard

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    pk = peaks()

    # ---- the step's matrices: N = 1: all 224 Llama-2-7B linears; N > 1: this rank's row shards of 16 70B layers
    if world == 1:
        shp = LLAMA2_7B_LAYER * N_LAYERS
        layer = LLAMA2_7B_LAYER
        total_job = sum(r * c for r, c in shp)
        workload, scaling = WORKLOAD, "weak"
    else:
        layer = []
        for (r, c) in LLAMA3_70B_LAYER:
            a, b = row_shard(r, world, rank, 128)
            layer.append((b - a, c))
        shp = layer * N_LAYERS_70B
        total_job = sum(r * c for r, c in LLAMA3_70B_LAYER) * N_LAYERS_70B
        workload, scaling = WORKLOAD_70B, "strong"
    sizes = [r * c for r, c in shp]
    total = sum(sizes)                                     # this rank's elements

    flat = torch.empty(total, dtype=torch.float32, device=device)
    gen = torch.Generator(device=device).manual_seed(1234 + rank)
    step_fill = 1 << 28
    for off in range(0, total, step_fill):
        flat[off:off + step_fill].normal_(0.0, 0.02, generator=gen)
    views, off = [], 0
    for (r, c), n in zip(shp, sizes):
        views.append(flat[off:off + n].view(r, c))
        off += n

    def step():
        # the batched public entry point: 16 matrices per launch
        if args.per_tensor:
            return [Q.quantize_4bit(v, blocksize=BLOCK, packed=True) for v in views]
        return Q.quantize_4bit_many(views, blocksize=BLOCK, packed=True)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # eager warm-up (loads the library, sets kernel attributes), then capture one step
    outs = step()
    torch.cuda.synchronize()
    del outs
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = step()
    for _ in range(args.warmup):
        graph.replay()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    job_elems = total_job                                  # whole-job elements per step (all ranks)
    value = job_elems * BYTES_PER_ELEM / (ms * 1e-3) / 1e9
    per_gpu = total * BYTES_PER_ELEM / (ms * 1e-3) / 1e9
    launches = args.steps * (len(views) if args.per_tensor else -(-len(views) // 16))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, rank, world, torch)
    del outs, graph
    torch.cuda.empty_cache()

    # ---- e2e: host buffers -> public API -> host results, copies inside the timed region
    host_in = [torch.empty(r, c, dtype=torch.float32).normal_(0.0, 0.02).pin_memory() for r, c in layer]
    host_out = [(torch.empty(r * c // 2, dtype=torch.uint8).pin_memory(),
                 torch.empty(r * c // BLOCK, dtype=torch.float32).pin_memory(),
                 torch.empty(r * c // BLOCK, dtype=torch.float32).pin_memory()) for r, c in layer]
    streams = [torch.cuda.Stream(device), torch.cuda.Stream(device)]
    big = max(r * c for r, c in layer)
    stage = [torch.empty(big, dtype=torch.float32, device=device) for _ in streams]
    n_rep = len(shp) // len(layer)

    def e2e_step():
        i = 0
        for _ in range(n_rep):
            for m, (r, c) in enumerate(layer):
                s = i % 2
                with torch.cuda.stream(streams[s]):
                    d = stage[s][:r * c].view(r, c)
                    d.copy_(host_in[m], non_blocking=True)
                    pkd, sc, zp = Q.quantize_4bit(d, blocksize=BLOCK, packed=True)
                    host_out[m][0].copy_(pkd, non_blocking=True)
                    host_out[m][1].copy_(sc, non_blocking=True)
                    host_out[m][2].copy_(zp, non_blocking=True)
                i += 1

    e2e_steps = max(1, min(args.steps, 3))
    e2e_step()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    e2e_value = job_elems * BYTES_PER_ELEM / e2e_s / 1e9
    h2d = total * 4
    d2h = total // 2 + 2 * (total // BLOCK) * 4
    launches += (1 + e2e_steps) * len(shp)
    del host_in, host_out, stage, flat, views
    torch.cuda.empty_cache()

    secondary = None
    if not args.no_secondary:
        if world == 1:
            secondary, n_l = secondary_single_gpu(device, pk, torch, Q)
            launches += n_l
        else:
            from tools.bench_tp_rows import tp_rows
            secondary = {"tp": tp_rows(device, rank, world, pk, torch, dist, Q)}

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample = one decoder layer
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        mats = cpu_sample()
        elems, times, threads, kind, what = time_cpu_reference(mats, 1, 3, 1)
        tcpu = min(times)
        _, ctimes, cthreads = time_cpu_c_port(mats, 3, 1)
        cpu = {"value": elems * BYTES_PER_ELEM / tcpu / 1e9, "unit": "GB/s", "cores": threads, "kind": kind,
               "sample": "one decoder layer (7 matrices, %d elements), best of 3; %s" % (elems, what),
               "c_port_value": elems * BYTES_PER_ELEM / min(ctimes) / 1e9, "c_port_threads": cthreads}

    if rank == 0:
        kernel = ("quantize_rows_tma_kernel<float,4,pack,A,blockwise>" if args.per_tensor
                  else "quantize_rows_tma_multi_kernel<float,4,pack>")
        tr = ncu_traffic("quantize_rows_tma_kernel" if args.per_tensor else "quantize_rows_tma_multi_kernel")
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "ours",
            "config": {"workload": workload, "elements_per_gpu": total, "elements_job": job_elems, "matrices_per_gpu": len(shp),
                       "blocksize": BLOCK, "bytes_per_element": BYTES_PER_ELEM,
                       "l2": "inputs (%.1f GB per GPU) larger than L2" % (total * 4 / 1e9),
                       "launch": ("%d per-matrix launches" % len(shp) if args.per_tensor else
                                  "quantize_4bit_many: %d multi-tensor launches (16 matrices each)" % -(-len(shp) // 16))
                                 + " replayed as one CUDA graph",
                       "parallelism": ("one GPU" if world == 1 else
                                       "row-sharded weights (row_shard(out, %d, rank, 128)), no data-path collective" % world)},
            "roofline": {"bound": "hbm", "kernel": kernel, "achieved": per_gpu, "peak": pk["hbm"],
                         "peak_source": pk["source"] + " hbm_gbs, burst copy", "unit": "GB/s", "frac": per_gpu / pk["hbm"],
                         "traffic": (tr["dram_bytes"] if tr else None),
                         "traffic_algorithmic": (tr.get("algorithmic_bytes") if tr else None),
                         "traffic_source": (tr["file"] + ": " + tr.get("launch", "") if tr else "no committed ncu capture found")},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "note": "per GPU: pinned host buffers, 2 streams, H2D + quantize + D2H per matrix"},
            "gpu_launches": launches,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary block (GEMM / dequantize / config 1 / TP rows)")
    ap.add_argument("--per-tensor", action="store_true", help="one quantize_4bit call (launch) per matrix instead of the batched entry")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
