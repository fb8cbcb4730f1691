"""Timeline of one bench step: the headline's quantize_4bit_many over all 224 Llama-2-7B linears (fp32 -> 4-bit
block-64 + pack, 14 launches of 16 matrices), captured in a CUDA graph like bench.py and replayed under
torch.profiler.  Prints one JSON line per launch of the profiled replay: start and device time in microseconds and
the gap to the next launch's start (negative when the next launch overlaps this one), then a summary line.

Usage: python tools/prof_quantize_step.py [--out DIR]   (--out: also write the trace and the JSON lines there)"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import quanta_b200 as Q

LAYER = [(4096, 4096)] * 4 + [(11008, 4096)] * 2 + [(4096, 11008)]      # bench.py LLAMA2_7B_LAYER
N_LAYERS = 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="directory for the trace and the per-launch lines")
    args = ap.parse_args()
    shp = LAYER * N_LAYERS
    total = sum(r * c for r, c in shp)
    flat = torch.empty(total, dtype=torch.float32, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(1234)
    for off in range(0, total, 1 << 28):
        flat[off:off + (1 << 28)].normal_(0.0, 0.02, generator=gen)
    views, off = [], 0
    for r, c in shp:
        views.append(flat[off:off + r * c].view(r, c))
        off += r * c

    outs = Q.quantize_4bit_many(views, blocksize=64, packed=True)
    torch.cuda.synchronize()
    del outs
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = Q.quantize_4bit_many(views, blocksize=64, packed=True)
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        graph.replay()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                 and "quantize_rows_tma" in e.name), key=lambda e: e.time_range.start)
    if not ev:
        sys.exit("no quantize_rows_tma launch in the trace")
    lines = []
    t0 = ev[0].time_range.start
    for i, e in enumerate(ev):
        nxt = ev[i + 1].time_range.start - e.time_range.end if i + 1 < len(ev) else None
        lines.append({"launch": i, "start_us": round(e.time_range.start - t0, 2),
                      "device_us": round(e.time_range.end - e.time_range.start, 2),
                      "gap_to_next_us": None if nxt is None else round(nxt, 2)})
    span = ev[-1].time_range.end - t0
    gaps = [l["gap_to_next_us"] for l in lines if l["gap_to_next_us"] is not None]
    lines.append({"summary": True, "device": torch.cuda.get_device_name(), "launches": len(ev),
                  "span_us": round(span, 1), "sum_device_us": round(sum(l["device_us"] for l in lines), 1),
                  "mean_gap_us": round(sum(gaps) / len(gaps), 2) if gaps else None, "kernel": ev[0].name})
    for l in lines:
        print(json.dumps(l))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        prof.export_chrome_trace(os.path.join(args.out, "quantize_step.pt.trace.json"))
        with open(os.path.join(args.out, "quantize_step.jsonl"), "w") as f:
            f.writelines(json.dumps(l) + "\n" for l in lines)


if __name__ == "__main__":
    main()
