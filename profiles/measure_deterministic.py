"""Cost of torch.use_deterministic_algorithms(True) for one TPAVIModule forward + backward (CUDA events after warm-up),
flag off and on alternated in the same process, at the shapes where the flag changes the work:
  * cfg2 Gram form (C = 256, N = 3 136, 128 sequences): no split there, so the two should be equal;
  * cfg2 token-space form (16 sequences): split token contractions and the batch-reduced dWz;
  * mode='embedded' at C = 256 (16 sequences): split dWz / dWcat;
  * C = 2048 with 3 views of 28 x 28 (2 sequences): dWcat in three K slices of 25 MB each;
  * Gram form with 4 sequences: the token contraction split 49 ways.
With the flag on, PyTorch also fills every torch.empty with NaN (fill_uninitialized_memory, its default); that is
part of what a user of the flag pays, so it is left on; a third arm turns it off
(torch.utils.deterministic.fill_uninitialized_memory = False) to separate the slab reductions from the NaN fill of the
blobs.  The device name and power limit are read in the same run.
Usage: python profiles/measure_deterministic.py [OUTDIR]   (writes OUTDIR/r03_deterministic.json; default profiles/)."""
from __future__ import annotations

import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from glfusion_b200 import TPAVIModule, tpavi  # noqa: E402

CASES = [  # name, mode, C, B, (T, H, W), dot algorithm (reserved[1] low byte)
    ("cfg2_gram_b128", "dot", 256, 128, (4, 28, 28), 2),
    ("cfg2_token_b16", "dot", 256, 16, (4, 28, 28), 1),
    ("embedded_c256_b16", "embedded", 256, 16, (4, 28, 28), 0),
    ("width2048_3views_b2", "dot", 2048, 2, (3, 28, 28), 0),
    ("gram_b4", "dot", 256, 4, (4, 28, 28), 2),
]
WARMUP, REPS, ROUNDS = 3, 10, 3


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in out.split(",")]
    except Exception:      # no nvidia-smi: the device name from torch, power limit unknown
        name, power, clk = torch.cuda.get_device_name(0), "unknown", "unknown"
    return name, power, clk


def timed(fn, det, fill=True):
    was = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(det)
    torch.utils.deterministic.fill_uninitialized_memory = fill
    try:
        for _ in range(WARMUP):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(REPS):
            fn()
        e1.record()
        torch.cuda.synchronize()
    finally:
        torch.use_deterministic_algorithms(was)
        torch.utils.deterministic.fill_uninitialized_memory = True
    return e0.elapsed_time(e1) / REPS


def module_step(mode, C, B, shape, algo, dev):
    torch.manual_seed(1)
    m = TPAVIModule(C, mode=mode).to(dev).train()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, C, *shape, generator=g).to(dev, torch.bfloat16).requires_grad_(True)
    dz = torch.randn(B, C, *shape, generator=g).to(dev, torch.bfloat16)

    def step():
        x.grad = None
        for p in m.parameters():
            p.grad = None
        old = tpavi.DOT_ALGO
        tpavi.DOT_ALGO = algo
        try:
            z, _ = m(x)
        finally:
            tpavi.DOT_ALGO = old
        z.backward(dz)
    return step


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles")
    os.makedirs(out_dir, exist_ok=True)
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda:0")
    name, power, clk = gpu_info()
    res = {"device": name, "power_limit": power, "max_sm_clock": clk,
           "method": f"TPAVIModule fwd+bwd, CUDA events, {WARMUP} warm-up + {REPS} timed steps per sample, flag off / on "
                     f"/ on without fill_uninitialized_memory alternated {ROUNDS} times in one process; median per arm (ms)",
           "cases": {}}
    for cname, mode, C, B, shape, algo in CASES:
        step = module_step(mode, C, B, shape, algo, dev)
        off, on, nofill = [], [], []
        for _ in range(ROUNDS):
            off.append(timed(step, False))
            on.append(timed(step, True))
            nofill.append(timed(step, True, fill=False))
        mo, mn, mf = statistics.median(off), statistics.median(on), statistics.median(nofill)
        res["cases"][cname] = {"mode": mode, "C": C, "B": B, "THW": list(shape), "dot_algo": algo,
                               "off_ms": [round(v, 4) for v in off], "on_ms": [round(v, 4) for v in on],
                               "off_median_ms": round(mo, 4), "on_median_ms": round(mn, 4),
                               "on_over_off": round(mn / mo, 4),
                               "on_nofill_ms": [round(v, 4) for v in nofill], "on_nofill_median_ms": round(mf, 4),
                               "on_nofill_over_off": round(mf / mo, 4)}
        print(cname, res["cases"][cname], flush=True)
        del step
        torch.cuda.empty_cache()
    path = os.path.join(out_dir, "r03_deterministic.json")
    with open(path, "w") as fh:
        json.dump(res, fh, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
