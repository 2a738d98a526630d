"""fp32 against bf16 parameters (``GlobalLocalFusion.to(torch.bfloat16)``) through the fused node
(forward_stacked, fwd + bwd, bf16 f4), replayed from CUDA graphs, the two arms alternating in one process.  A bf16 block
adds one launch forward (the fp32 parameter copy) and one backward (the gradients rounded to bf16) per block; everything
else is the fp32-parameter path, so the time should differ by those four short passes.

Shapes: the bench shape (8 clips = 128 frames x 4 views x 28 x 28 tokens, C = 256: 205 MB per activation, larger than
the 126 MB L2) and the width2048 shape of bench.py (8 frames x 3 views x 28 x 28, C = 2048).
Writes profiles/r04_half_params.json (or the path given as argv[1]): ms per step of each arm, the bf16 / fp32 ratio,
the kernel launches of one step (torch.profiler, CUDA activity), the GPU name and its power limit."""
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
from profiles.measure_fp16 import launches, time_graph  # noqa: E402


def setup(pdt, C, V, B, dev):
    f = bench.seeded_fusion(C, dev).to(pdt)
    g = torch.Generator().manual_seed(5)
    f4 = [torch.randn(B, C, bench.HH, bench.WW, generator=g).to(dev, torch.bfloat16).requires_grad_(True)
          for _ in range(V)]
    cl = [torch.randn(B, bench.NCLS, bench.HH, bench.WW, generator=g).to(dev) for _ in range(V)]
    ct = [torch.randn(B, 1, bench.HH, bench.WW, generator=g).to(dev) for _ in range(V)]
    dz = torch.randn(B, V, bench.HH, bench.WW, C, generator=g).to(dev, torch.bfloat16).permute(0, 4, 1, 2, 3)
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


def measure(name, C, V, B, reps, rounds, dev):
    arms = {}
    for pdt in (torch.float32, torch.bfloat16):
        step, graph = setup(pdt, C, V, B, dev)
        arms[pdt] = {"graph": graph, "ms": [], "launches": launches(step, dev)}
    for _ in range(rounds):                     # alternate the two arms, many short windows each
        for pdt in (torch.float32, torch.bfloat16):
            arms[pdt]["ms"].append(time_graph(arms[pdt]["graph"], reps, dev))
    f32, b16 = arms[torch.float32], arms[torch.bfloat16]
    mf, mb = statistics.median(f32["ms"]), statistics.median(b16["ms"])
    return {"workload": name, "C": C, "views": V, "frames": B, "tokens": B * V * bench.HH * bench.WW,
            "ms_per_step_fp32_params": round(mf, 4), "ms_per_step_bf16_params": round(mb, 4),
            "ratio_bf16_over_fp32": round(mb / mf, 4),
            "ms_fp32_params_all": [round(x, 4) for x in f32["ms"]], "ms_bf16_params_all": [round(x, 4) for x in b16["ms"]],
            "launches_fp32_params": f32["launches"], "launches_bf16_params": b16["launches"],
            "timing": f"median of {rounds} alternating windows of {reps} CUDA-graph replays per arm"}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r04_half_params.json")
    assert torch.cuda.is_available(), "measure_half_params.py needs a GPU"
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
