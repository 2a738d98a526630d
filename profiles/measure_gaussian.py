"""TPAVIModule(mode='gaussian') forward + backward timed with CUDA events after warm-up, against
  * mode='embedded' on the same shapes (same attention kernels, theta / phi projected and used), and
  * the oracle's literal gaussian forward + backward (oracle/tpavi_oracle.py: tpavi_fwd_bwd) in PyTorch eager under
    torch.autocast(bfloat16) on the same GPU.
Shapes: C = 128 (flash kernels, (DQK, DV) = (128, 64)) and cfg2's C = 256 at N = 3 136 tokens (chunked exact path).

FLOPs of the algorithm executed per sequence (attention only): forward 2 N^2 (C + C'); backward with recompute
4 N^2 C + 4 N^2 C' + 4 N^2 C + 2 N^2 C'.  The device name and its power limit are read in the same run.
Usage: python profiles/measure_gaussian.py [OUTDIR]   (writes OUTDIR/measure_gaussian.json; default profiles/)."""
from __future__ import annotations

import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from glfusion_b200 import TPAVIModule  # noqa: E402
from oracle import tpavi_oracle as O  # noqa: E402

SHAPES = [  # C, B, (T, H, W)
    (128, 16, (4, 28, 28)),
    (256, 16, (4, 28, 28)),
]
WARMUP, REPS = 5, 20


def attn_flops(B, N, C, Ci):
    fwd = 2 * N * N * (C + Ci)
    bwd = 4 * N * N * C + 4 * N * N * Ci + 4 * N * N * C + 2 * N * N * Ci
    return B * fwd, B * bwd


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except Exception:      # no nvidia-smi: the device name from torch, power limit unknown
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def timed(fn, dev):
    for _ in range(WARMUP):
        fn()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPS):
        fn()
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / REPS


def module_step(mode, C, B, shape, dev):
    torch.manual_seed(1)
    m = TPAVIModule(C, mode=mode).to(dev).train()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, C, *shape, generator=g).to(dev, torch.bfloat16).requires_grad_(True)
    dz = torch.randn(B, C, *shape, generator=g).to(dev, torch.bfloat16)

    def step():
        x.grad = None
        for p in m.parameters():
            p.grad = None
        z, _ = m(x)
        z.backward(dz)
    return step


def oracle_step(C, B, shape, dev):
    p = {k: (v.to(dev) if v.is_floating_point() else v.to(dev)) for k, v in O.init_params(C, seed=1,
                                                                                            randomize_affine=True).items()}
    g = torch.Generator().manual_seed(2)
    x = torch.randn(B, C, *shape, generator=g).to(dev)
    dz = torch.randn(B, C, *shape, generator=g).to(dev)

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            O.tpavi_fwd_bwd(x, dz, p, mode="gaussian", training=True)
    return step


def main():
    out_dir = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles")
    if not torch.cuda.is_available():
        raise SystemExit("measure_gaussian.py needs a CUDA device (no CPU timing is reported)")
    dev = torch.device("cuda:0")
    name, power = gpu_info()
    rows = []
    for C, B, shape in SHAPES:
        N = shape[0] * shape[1] * shape[2]
        Ci = C // 2
        ff, fb = attn_flops(B, N, C, Ci)
        r = dict(C=C, Ci=Ci, B=B, N=N, path="flash" if C <= 128 else "chunked",
                 attn_gflop_fwd=ff / 1e9, attn_gflop_bwd=fb / 1e9)
        r["gaussian_ms"] = timed(module_step("gaussian", C, B, shape, dev), dev)
        r["embedded_ms"] = timed(module_step("embedded", C, B, shape, dev), dev)
        r["oracle_autocast_ms"] = timed(oracle_step(C, B, shape, dev), dev)
        r["gaussian_attn_tflops_lower_bound"] = (ff + fb) / (r["gaussian_ms"] * 1e-3) / 1e12   # whole block's time
        rows.append(r)
        print(json.dumps(r))
    res = dict(device=name, power_limit=power, warmup=WARMUP, reps=REPS, rows=rows,
               note="fwd+bwd of one block per step, CUDA events; attention FLOPs over the whole block's time")
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "measure_gaussian.json"), "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(dict(device=name, power_limit=power)))


if __name__ == "__main__":
    main()
