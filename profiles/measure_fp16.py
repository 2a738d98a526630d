"""fp16 against bf16 f4 through the fused node (GlobalLocalFusion.forward_stacked, fwd + bwd), replayed from CUDA graphs,
the two dtypes alternating in one process.  fp16 is an I/O dtype: the boundary kernels read and write 2-byte elements in
both, so the bytes, the launches and the time should match.

Shapes: the bench shape (8 clips = 128 frames x 4 views x 28 x 28 tokens, C = 256: 205 MB per activation, larger than
the 126 MB L2) and the width2048 shape of bench.py (8 frames x 3 views x 28 x 28, C = 2048).
Writes profiles/r03_fp16.json (or the path given as argv[1]): ms per step of each dtype, the fp16 / bf16 ratio, the
kernel launches of one step (torch.profiler, CUDA activity), the GPU name and its power limit."""
from __future__ import annotations

import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def setup(dt, C, V, B, dev):
    f = bench.seeded_fusion(C, dev)
    g = torch.Generator().manual_seed(5)
    f4 = [torch.randn(B, C, bench.HH, bench.WW, generator=g).to(dev).to(dt).requires_grad_(True) for _ in range(V)]
    cl = [torch.randn(B, bench.NCLS, bench.HH, bench.WW, generator=g).to(dev) for _ in range(V)]
    ct = [torch.randn(B, 1, bench.HH, bench.WW, generator=g).to(dev) for _ in range(V)]
    dz = torch.randn(B, V, bench.HH, bench.WW, C, generator=g).to(dev).to(dt).permute(0, 4, 1, 2, 3)
    params = [p for p in f.parameters() if p.requires_grad]

    def step():
        for t in f4:
            t.grad = None
        for p in params:
            p.grad = None
        f.forward_stacked(f4, cl, ct).backward(dz)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize(dev)
    return step, graph


def time_graph(graph, reps, dev):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def launches(step, dev):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize(dev)
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


def measure(name, C, V, B, reps, rounds, dev):
    arms = {}
    for dt in (torch.bfloat16, torch.float16):
        step, graph = setup(dt, C, V, B, dev)
        arms[dt] = {"step": step, "graph": graph, "ms": [], "launches": launches(step, dev)}
    for _ in range(rounds):                     # alternate the two dtypes, many short windows each
        for dt in (torch.bfloat16, torch.float16):
            arms[dt]["ms"].append(time_graph(arms[dt]["graph"], reps, dev))
    bf, hf = arms[torch.bfloat16], arms[torch.float16]
    mb, mh = statistics.median(bf["ms"]), statistics.median(hf["ms"])
    return {"workload": name, "C": C, "views": V, "frames": B, "tokens": B * V * bench.HH * bench.WW,
            "ms_per_step_bf16": round(mb, 4), "ms_per_step_fp16": round(mh, 4), "ratio_fp16_over_bf16": round(mh / mb, 4),
            "ms_bf16_all": [round(x, 4) for x in bf["ms"]], "ms_fp16_all": [round(x, 4) for x in hf["ms"]],
            "launches_bf16": bf["launches"], "launches_fp16": hf["launches"],
            "timing": f"median of {rounds} alternating windows of {reps} CUDA-graph replays per dtype"}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_fp16.json")
    assert torch.cuda.is_available(), "measure_fp16.py needs a GPU"
    dev = torch.device("cuda:0")
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:          # the numbers still stand with the torch device name
        q = f"nvidia-smi unavailable: {exc!r}"
    res = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": q,
           "bench_shape": measure("bench shape: 8 clips x 16 frames, 4 views x 28x28, C=256 (Gram form)", 256, bench.V,
                                  8 * bench.F, reps=20, rounds=15, dev=dev),
           "width2048": measure("width2048: 8 frames, 3 views x 28x28, C=2048 (token-space form)", 2048, 3, 8,
                                reps=10, rounds=10, dev=dev)}
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if not kk.endswith("_all")})
                      for k, v in res.items()}, indent=1))


if __name__ == "__main__":
    main()
