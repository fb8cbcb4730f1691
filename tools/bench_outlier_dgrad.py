"""Input gradient of the outlier-split Linear8bitLt, dx[M,K] = dy[M,N] . W16[N,K] with
W16 = round_act(qw / cw), on the OPT-6.7B layer shapes of tools/bench_outlier.py.  Per point three variants
are timed in the same process, alternating, by CUDA-graph replay over rotating weight copies (footprint
> 400 MB, so weights stream from HBM on every call), CUDA events:

  fused    int8_outlier_dgrad (the fused dequantize-transposed GEMM, int8 row-wise codes)
  unfused  (qw.float() / cw[:, None]).to(bf16) + torch.matmul(dy, W16)
  w8a16    linear_wna16_dgrad(bits=8, blocksize=64) on the same shape: the same 8-bit code stream with
           a scale and a zero-point per 64 codes instead of one multiplier per row

Roof of the fused kernel: bytes N*K + 4N + 2MN + 2MK over 7.7 TB/s, flops 2MNK over 2,250 TFLOP/s (HGX
B200 data sheet, one GPU, dense BF16, 1,000 W); the binding one is reported.  The card's name and power
limit are read in the same call and written to every line.

    python tools/bench_outlier_dgrad.py --out profiles/r06_bench_outlier_dgrad.jsonl"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import quanta_b200 as Q
from quanta_b200.nn import int8_outlier_dgrad, linear_wna16_dgrad, rowwise_quantize_sym

HBM_BPS, TC_FLOPS = 7.7e12, 2.25e15

ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--ms", default="1,16,64,256,1024,4096")
ap.add_argument("--shapes", default="4096x4096,16384x4096,4096x16384", help="NxK: out_features x in_features")
ap.add_argument("--rounds", type=int, default=5, help="alternating timed replays per variant")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("bench_outlier_dgrad.py needs a CUDA device")

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
card = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}
dt = torch.bfloat16
lines = []


def time_graphs(graphs, calls):
    """Median microseconds per call of each graph, replays alternating between the graphs."""
    samples = [[] for _ in graphs]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for i, g in enumerate(graphs):
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            samples[i].append(e0.elapsed_time(e1) * 1e3 / calls)
    return [statistics.median(s) for s in samples]


def capture(fn, calls):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(2):
            fn(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        keep = [fn(i) for i in range(calls)]
    g.replay()
    torch.cuda.synchronize()
    return g, keep


for (N, K) in [tuple(int(v) for v in sh.split("x")) for sh in args.shapes.split(",")]:
    wbytes = N * K + 4 * N
    copies = max(8, int(400e6 // wbytes) + 1)
    rows, w8 = [], []
    for i in range(copies):
        w = torch.randn(N, K, device="cuda") * 0.02
        rows.append(rowwise_quantize_sym(w))
        w8.append(Q.quantize_8bit(w, blocksize=64))
        del w
    for M in [int(v) for v in args.ms.split(",")]:
        dy = torch.randn(M, N, device="cuda").to(dt)
        fused = lambda i: int8_outlier_dgrad(dy, *rows[i % copies])
        unfused = lambda i: torch.matmul(dy, (rows[i % copies][0].float() / rows[i % copies][1][:, None]).to(dt))
        w8a16 = lambda i: linear_wna16_dgrad(dy, *w8[i % copies], bits=8, blocksize=64, out_features=N, in_features=K)
        graphs, keeps = [], []
        for fn in (fused, unfused, w8a16):
            g, keep = capture(fn, copies)
            graphs.append(g)
            keeps.append(keep)
        us_fused, us_unfused, us_w8 = time_graphs(graphs, copies)
        flops = 2.0 * M * N * K
        abytes = wbytes + 2 * M * N + 2 * M * K
        t_hbm, t_tc = abytes / HBM_BPS * 1e6, flops / TC_FLOPS * 1e6
        line = {"op": "int8_outlier_dgrad", "N": N, "K": K, "M": M, "dtype": "bf16",
                "us_fused": round(us_fused, 2), "us_unfused": round(us_unfused, 2), "us_w8a16_dgrad": round(us_w8, 2),
                "unfused_over_fused": round(us_unfused / us_fused, 2), "fused_over_w8a16": round(us_fused / us_w8, 3),
                "bound": "hbm" if t_hbm >= t_tc else "tensor", "frac_of_roof": round(max(t_hbm, t_tc) / us_fused, 3),
                "t_hbm_us": round(t_hbm, 2), "t_tensor_us": round(t_tc, 2), "calls_per_replay": copies, **card}
        print(json.dumps(line), flush=True)
        lines.append(line)
        del graphs, keeps
    del rows, w8
    torch.cuda.empty_cache()
if args.out:
    with open(args.out, "w") as f:
        for l in lines:
            f.write(json.dumps(l) + "\n")
