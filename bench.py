#!/usr/bin/env python
"""bench.py — GL-Fusion fusion hot path (gate+concat -> MGFM + MLFM -> sum) forward+backward throughput on B200.

    python bench.py --gpus 1 --steps 20 --warmup 5            # our arm (libglf_sm100a.so)
    python bench.py --impl reference --steps 3 --warmup 1     # the reference algorithm on the host CPU cores
    python bench.py --steps 20 --dump-outputs DIR              # + the last timed step's output and gradients as .npy

Workload = BASELINE.json configs[1]: MGFM+MLFM modules only, 4 views x 16 frames x 28x28 tokens, C=256, bf16,
fwd+bwd, frames-as-batch layout (Global_and_Local, R/models/ours.py:1819-1821): one clip = 16 sequences of
4*28*28 = 3136 tokens.  A step processes `--clips` clips per GPU (default 8 -> 128 sequences, 205 MB of bf16 features,
larger than the 126 MB L2, so no L2 flush is needed between iterations).

One JSON line on stdout (rank 0).  Under torchrun (N>1) clips are sharded by rank (weak scaling: fixed clips/GPU), the
only collective is the all-reduce of the fusion-weight gradients.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

V, F, HH, WW = 4, 16, 28, 28
NCLS = 5


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "bf16_tflops_burst": float(d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "bf16_tflops_burst": 1590.0, "source": "fallback"}


class ClockSampler:
    """SM clock / throttle-reason sampling DURING the timed region: an NVML polling thread (5 ms period) in this
    process; `nvidia-smi -lms` as the fallback when NVML cannot be loaded."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None
        self.nvml = None
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, h

    def _poll(self, nv, h):
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(h))
                for bit, name in self.BITS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            nv, h = self._nvml_handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.nvml = nv
            self.th = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.th.join(timeout=1)
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------------------------
def make_inputs(clips: int, C: int, seed: int, device, pinned: bool = False):
    B = clips * F
    g = torch.Generator().manual_seed(seed)
    f4 = [torch.randn(B, C, HH, WW, generator=g).to(torch.bfloat16) for _ in range(V)]
    cls = [torch.randn(B, NCLS, HH, WW, generator=g) for _ in range(V)]
    ctr = [torch.randn(B, 1, HH, WW, generator=g) for _ in range(V)]
    if pinned:
        return [t.pin_memory() for t in f4], [t.pin_memory() for t in cls], [t.pin_memory() for t in ctr]
    return [t.to(device) for t in f4], [t.to(device) for t in cls], [t.to(device) for t in ctr]


def randomize_affine_(module, seed: int):
    """SURVEY F3: BatchNorm gamma / beta are initialised to 0 in the reference (the attention branch then outputs 0 and
    its gradients vanish), so a benchmark on "random-init" weights re-randomises the BN and LayerNorm affines."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p, mean in ((module.W_z[1].weight, 1.0), (module.W_z[1].bias, 0.0), (module.norm_layer.weight, 1.0),
                        (module.norm_layer.bias, 0.0)):
            p.copy_(mean + 0.2 * torch.randn(p.shape, generator=g))


def seeded_fusion(C: int, device):
    from glfusion_b200 import GlobalLocalFusion
    torch.manual_seed(0)
    f = GlobalLocalFusion(in_channels=C)     # the reference's own initialisers (identical RNG stream, tests/test_module_cpu.py)
    randomize_affine_(f.global_attn, 10)
    randomize_affine_(f.local_attn, 11)
    return f.to(device).train()


def dot_algorithm(C: int) -> str:
    """Which exact reassociation of mode='dot' libglf_sm100a runs for the bench shape (glf_api.cu: make_dims):
    the Gram form when the sequences are long against the channel count (N >= 3 C at C = 256 where the per-sequence
    chain kernels exist, 5 C below, 8 C above), unless GLF_DOT_ALGO pins it."""
    pin = int(os.environ.get("GLF_DOT_ALGO", "0"))
    if pin in (1, 2):
        return "token" if pin == 1 else "gram"
    thr = 3 if (C == 256 and os.environ.get("GLF_GRAM_CHAIN", "1") != "0") else (8 if C > 256 else 5)
    return "gram" if V * HH * WW >= thr * C else "token"


def algorithmic_work(clips: int, C: int):
    """FLOPs of the algorithm actually executed, per step (both modules, fwd+bwd)."""
    N = V * HH * WW
    rows = clips * F * N
    Ci = C // 2
    if dot_algorithm(C) == "gram":
        # token-sized products: S = X^T X, U = X Q^T (fwd); R = dV^T X, dX = [dV | X][E ; F] (bwd) = 10 rows C^2;
        # per-sequence [C x C] chain: 3 C^3 forward + 12 C^3 backward (in units of 2 C^3 FLOPs: 1.5 + 6)
        big = 2 * rows * C * C * 5
        small = clips * F * 15 * C * C * C
        return 2 * (big + small), rows
    # token-space form (W' = Wz M^T folded in)
    fwd = 2 * rows * C * 3 * Ci + 2 * rows * Ci * Ci + 2 * rows * Ci * C
    bwd = 2 * rows * C * Ci * 2 + 2 * rows * Ci * Ci * 2 + 2 * rows * 3 * Ci * C * 2
    small = clips * F * (2 * C * Ci * Ci) * 3
    return 2 * (fwd + bwd + small), rows


def bind_to_gpu_numa(index: int, world: int = 1):
    """Pin this process to the CPUs NVML reports as local to GPU `index`, so that the pinned host staging buffers of
    the end-to-end pipeline are allocated on the GPU's own NUMA node (8 ranks otherwise contend for one socket's
    memory and PCIe root).  Returns (original affinity, number of local CPUs) or (None, None)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        ncpu = os.cpu_count() or 1

        def cpus_of(handle):
            mask = pynvml.nvmlDeviceGetCpuAffinity(handle, (ncpu + 63) // 64)
            return [i for i in range(ncpu) if (int(mask[i // 64]) >> (i % 64)) & 1]
        cpus = cpus_of(h)
        orig = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in orig]
        note = "NVML affinity"
        if world > 1 and cpus:
            # when NVML reports the SAME CPU set for every GPU (one NUMA node for the whole box) binding all ranks to
            # it would stack them on the same cores: each rank takes its own slice of the set instead.  The pinned
            # staging memory of all ranks then still comes from that one node - a platform limit, stated in the line.
            same = True
            for i in range(pynvml.nvmlDeviceGetCount()):
                if i != index and cpus_of(pynvml.nvmlDeviceGetHandleByIndex(i)) != cpus_of(h):
                    same = False
            if same:
                per = max(1, len(cpus) // world)
                cpus = cpus[(index % world) * per:(index % world) * per + per] or cpus
                note = "one CPU set for all GPUs (single NUMA node): ranks take disjoint slices of it"
        if cpus:
            os.sched_setaffinity(0, cpus)
            return orig, len(cpus), note
    except Exception:
        pass
    return None, None, None


DUMP_BYTES = 60_000_000


def dump_outputs(path: str, arrays: dict) -> None:
    """Write each tensor as <path>/<name>.npy in float32, in all at most DUMP_BYTES.  Arrays are served smallest
    first; one larger than its even share of what is left is replaced by a seeded sample of its flattened (logical,
    row-major) elements.  The sample depends only on the array's shape, so two builds dump the same positions."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES // 4
    items = sorted(arrays.items(), key=lambda kv: (kv[1].numel(), kv[0]))
    for i, (name, t) in enumerate(items):
        t = t.detach()
        k = min(t.numel(), left // (len(items) - i))
        left -= k
        if k < t.numel():
            idx = torch.randint(0, t.numel(), (k,), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    from glfusion_b200 import dp
    rank, local_rank, world = dp.init_process_group("nccl")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    orig_affinity, numa_cpus, numa_note = bind_to_gpu_numa(local_rank, world)
    C = args.channels
    clips = args.clips
    fusion = seeded_fusion(C, dev)
    f4, cls, ctr = make_inputs(clips, C, 100 + rank, dev)
    for t in f4:
        t.requires_grad_(True)
    B = clips * F
    dz = torch.randn(B, V, HH, WW, C, device=dev, dtype=torch.bfloat16,
                     generator=torch.Generator(device=dev).manual_seed(0)).permute(0, 4, 1, 2, 3)
    bucket = dp.GradBucket(list(fusion.global_attn._plist()) + list(fusion.local_attn._plist()))
    bucket.bind([fusion.global_attn, fusion.local_attn])   # gradients are written into the all-reduce bucket directly
    # the fusion-weight gradient average as one kernel over NVLink peer memory (NCCL stays the fallback)
    p2p = bool(world > 1 and args.p2p_allreduce and bucket.enable_p2p())
    # (the side-stream launch must be joined inside the same capture: only when the exchange is captured with the step)
    overlap = bool(p2p and args.overlap_allreduce and (not args.graph or args.graph_allreduce != 0))
    if overlap:
        bucket.overlap_with(fusion)      # the exchange starts before the gate backward, on a side stream

    params = [p for p in fusion.parameters() if p.requires_grad]
    last = {}                            # --dump-outputs: the step's forward output (a graph replay rewrites it in place)

    def compute():
        for t in f4:
            t.grad = None
        for p in params:
            p.grad = None                # optimizer.zero_grad(set_to_none=True): gradients are assigned, not accumulated
        out = fusion.forward_stacked(f4, cls, ctr)
        out.backward(dz)
        if args.dump_outputs:
            last["out"] = out.detach()   # without the autograd graph, which must not outlive the step

    graph = None
    allreduce_in_graph = False
    if args.graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                compute()
                if world > 1:
                    bucket.allreduce_mean()      # also brings the NCCL communicator up before any capture
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        if world > 1 and (args.graph_allreduce == 1 or (args.graph_allreduce < 0 and p2p)):
            # the gradient all-reduce is captured with the step: one graph launch per step, no host gap between the
            # last backward kernel and the NCCL kernel.  Any capture problem falls back to an eager all-reduce.
            try:
                g2 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g2):
                    compute()
                    bucket.allreduce_mean()
                graph, allreduce_in_graph = g2, True
            except Exception as exc:           # noqa: BLE001
                log(f"all-reduce capture failed ({exc!r}); using an eager all-reduce after the graph")
                torch.cuda.synchronize()
        if graph is None:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                compute()

    def run_step():
        if graph is not None:
            graph.replay()
        else:
            compute()
        if world > 1 and not allreduce_in_graph:
            bucket.allreduce_mean()      # the only collective: fusion-weight gradients over NVLink (peer kernel / NCCL)

    for _ in range(max(args.warmup, 3)):
        run_step()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(nsteps):
        torch.cuda.synchronize()
        e0.record()
        for _ in range(nsteps):
            run_step()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()
        return dp.max_over_ranks(e0.elapsed_time(e1) / nsteps, device=dev)

    # B200 power management: after ~50 ms of this load the board reaches its software power cap and the SM clock drops
    # from 1965 MHz to ~1.7 GHz (NVML: sw_power_cap).  A cold K-step burst is therefore ~8 % faster than the same steps
    # in steady state, and data-parallel ranks (which wait for each other every step) always run at the steady-state
    # pace.  `value` is the steady-state figure at every N: the burst is timed first and reported beside it, then
    # `settle_ms` of untimed steps bring the board to its sustained clocks before the K timed steps.
    burst_ms = timed(args.steps)
    settle_steps = 0
    if args.settle_ms > 0:
        nset = max(1, int(args.settle_ms / max(burst_ms, 1e-3)))
        for _ in range(nset):
            run_step()
        settle_steps = nset
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms = timed(args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        arrays = {"out": last["out"]}
        arrays.update({f"grad_f4_{v}": t.grad for v, t in enumerate(f4)})
        arrays.update({"grad_" + n: p.grad for n, p in fusion.named_parameters() if p.grad is not None})
        dump_outputs(args.dump_outputs, arrays)

    # ---- end-to-end: host (pinned) inputs -> H2D -> fwd+bwd -> D2H of the step's scalar result ----------------------
    hf4, hcls, hctr = make_inputs(clips, C, 100 + rank, dev, pinned=True)
    res_host = torch.zeros(1, dtype=torch.float32).pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in hf4 + hcls + hctr)

    # double-buffered input pipeline: while step i computes, the copy stream moves step i+1's inputs host -> device
    # into a staging set; the compute stream then takes them with one device-to-device copy (the CUDA graph reads
    # fixed addresses).  Every timed step contains one full H2D input copy and one D2H result read.
    dev_inputs = [t.detach() for t in f4 + cls + ctr]
    host_inputs = hf4 + hcls + hctr
    staging = [torch.empty_like(t) for t in dev_inputs]
    copy_stream = torch.cuda.Stream()
    copy_done = torch.cuda.Event()
    staged_free = torch.cuda.Event()

    def issue_h2d():
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(staged_free)
            for dst, src in zip(staging, host_inputs):
                dst.copy_(src, non_blocking=True)
            copy_done.record(copy_stream)

    def e2e_step():
        cur = torch.cuda.current_stream()
        cur.wait_event(copy_done)
        for dst, src in zip(dev_inputs, staging):
            dst.copy_(src, non_blocking=True)
        staged_free.record(cur)
        issue_h2d()                       # next step's inputs, overlapped with this step's compute
        run_step()
        res_host.copy_(f4[0].grad.float().abs().mean().reshape(1), non_blocking=True)

    staged_free.record(torch.cuda.current_stream())
    issue_h2d()
    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    e0.record()
    esteps = args.steps
    for _ in range(esteps):
        e2e_step()
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = dp.max_over_ranks(e0.elapsed_time(e1) / esteps, device=dev)

    if rank != 0:
        return
    flops, rows = algorithmic_work(clips, C)
    pk = peaks()
    total_clips = clips * world
    value = total_clips / (ms * 1e-3)
    out = {
        "metric": "fusion fwd+bwd clips/sec", "value": round(value, 2), "unit": "clips/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: MGFM+MLFM modules only, 4 views x 16 frames x 28x28 tokens, "
                               f"C={C}, bf16 fwd+bwd, frames-as-batch (B={clips * F} sequences x N={V * HH * WW} tokens per GPU)",
                   "clips_per_gpu_per_step": clips, "mode": "dot", "dot_algorithm": dot_algorithm(C),
                   "cuda_graph": bool(args.graph), "allreduce_in_graph": allreduce_in_graph,
                   "allreduce": ("none (1 GPU)" if world == 1 else
                                 ("glf_p2p_allreduce kernel over NVLink peer memory" +
                                  (", launched from the backward pass beside the gate backward" if overlap else "")
                                  if p2p else "NCCL all_reduce(AVG)")),
                   "l2": "inputs (%.0f MB/step) exceed the 126 MB L2; no flush" % (rows * C * 2 / 1e6),
                   "e2e_pipeline": "pinned host inputs; H2D of step i+1 on a copy stream overlaps compute of step i",
                   "parallelism": f"dp{world}",
                   "settle": f"{settle_steps} untimed steps (~{args.settle_ms:.0f} ms) before the timed region: steady-state "
                             "clocks under the software power cap at every N"},
        "e2e": {"value": round(total_clips / (e2e_ms * 1e-3), 2), "unit": "clips/s",
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4},
        "gpu_launches": None,
        "clocks": clocks,
        "burst": {"value": round(total_clips / (burst_ms * 1e-3), 2), "unit": "clips/s", "ms_per_step": round(burst_ms, 4),
                  "note": "the same K steps timed right after warm-up, before the board reaches its power cap"},
        "achieved_tflops_algorithmic": round(flops / (ms * 1e-3) / 1e12, 2),
        "peaks": pk,
    }
    # roofline = the dominant kernel BY TIME PER KERNEL NAME of the step (profiles/r02_*_launches.csv): the big K-major
    # tile GEMM that forms dX (two launches per step); the largest single launch (fused LayerNorm backward pair) and the
    # largest tensor-core product (S = X^T X) are reported beside it, and the whole step against its HBM floor.
    ln = kernel_probe(args, dev, clips, C, pk)["roofline"]
    if dot_algorithm(C) == "gram":
        gm = dx_gemm_probe(dev, clips, C, pk)
        gm["launches_per_step"] = 2
        ln["launches_per_step"] = 1
        sec = gram_probe(dev, clips, C, pk)
        gr = gram_family_probe(dev, clips, C, pk, sec["ms_per_launch"])
        fam = {"roofline_dx_gemm": gm, "roofline_ln_bwd": ln, "roofline_gram": gr}
        if C == 256:
            ug = u_gemm_probe(dev, clips, C, pk)
            ug["launches_per_step"] = 2
            fam["roofline_u_gemm"] = ug
        for v in fam.values():
            v["share_of_step"] = round(v["launches_per_step"] * v["ms_per_launch"] / burst_ms, 3)
            v["share_note"] = "launches_per_step x ms_per_launch / burst ms_per_step (both timed at boost clocks)"
        top = max(fam, key=lambda k: fam[k]["share_of_step"])      # dominant kernel by time per kernel name
        out["roofline"] = dict(fam[top], selected="largest launches_per_step x ms_per_launch of " + ", ".join(sorted(fam)))
        out.update(fam)
        out["roofline_secondary"] = sec
        # the algorithm that runs (DESIGN.md section 2, Gram form): gate 3P + 2 x (S 1P + U 2P) + LN pair 5P forward,
        # LN pair 7P + 2 x (R 2P + dX 3P) + gate 4P backward = 35 passes of P = rows x C x 2 bytes
        step_bytes = 35 * rows * C * 2
        out["roofline_step"] = {
            "bound": "hbm", "executed_bytes_per_step": step_bytes, "passes": 35,
            "achieved": round(step_bytes / (ms * 1e-3) / 1e9, 1), "achieved_burst": round(step_bytes / (burst_ms * 1e-3) / 1e9, 1),
            "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": round(step_bytes / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], 4),
            "frac_burst": round(step_bytes / (burst_ms * 1e-3) / 1e9 / pk["hbm_gbs"], 4),
            "note": "token-sized activation passes only; the per-sequence [C x C] matrices (1/12 of a pass each) are not counted"}
    else:
        out["roofline"] = ln
    out["gpu_launches"] = (count_launches(clips, C) + (1 if p2p else 0)) * args.steps
    out["e2e"]["per_gpu"] = round(out["e2e"]["value"] / world, 2)
    out["config"]["host_numa"] = (f"process bound to {numa_cpus} CPUs local to its GPU ({numa_note})"
                                  if numa_cpus else "no NUMA binding")
    if orig_affinity is not None:
        os.sched_setaffinity(0, orig_affinity)       # the CPU baseline below uses every host core again
    if world == 1 and not args.no_width2048:
        try:
            out["width2048"] = width2048(dev, pk)
        except Exception as exc:       # noqa: BLE001  (a secondary object must not take the bench line down)
            out["width2048"] = {"unavailable": repr(exc)[:200]}
        torch.cuda.empty_cache()
    if world == 1 and not args.no_gpu_reference:
        out["gpu_reference"] = gpu_reference(C, dev)
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline(C, seconds=args.cpu_seconds)
    emit(out)


def count_launches(clips: int, C: int) -> int:
    """Kernels launched by libglf_sm100a per step (fwd+bwd, both modules + gate), counted from the orchestration in
    glfusion_b200/csrc/glf_api.cu (memset/memcpy nodes excluded); agrees with profiles/r01_v11_launches.csv (39,
    token-space form), profiles/r01_v17_launches.csv (55, Gram form as batched tile GEMMs) and
    profiles/r02_v3_launches.csv / r02_v8_launches.csv (27, Gram form with the per-sequence chain kernels; 25 since the weight
    preparation rides along in the S launch)."""
    if dot_algorithm(C) == "gram" and C == 256 and os.environ.get("GLF_GRAM_CHAIN", "1") != "0":
        fwd_mod = 4      # S (gram_kernel; the weight preparation rides along as extra CTAs), chain_fwd, U GEMM, bn_finalize
        bwd_mod = 6      # finalize, R (gram_kernel), chain_bwd, wgrad, wgrad_reduce, dX GEMM
    elif dot_algorithm(C) == "gram":
        fwd_mod = 8 if C == 128 else 9   # (prep_weights,) S, T, M, W', Q~ GEMMs, cvec, U GEMM, bn_finalize
        bwd_mod = 16     # finalize, R (gram_kernel), kprep, dQ~, dW', dW~theta, dWz, dM, dW~g, dT, dW~phi, G0, H GEMMs,
        #                  assemble_F, dX GEMM, unpack_grads
    else:
        fwd_mod = 6      # prep_weights, proj GEMM, M GEMM, W' GEMM, U GEMM, bn_finalize
        bwd_mod = 11     # finalize, apply, dTheta, dW', dWz, dM, dPhi, dG, dWcat, dX, bias-gradient reduction
    pair = 2             # fused MGFM+MLFM LayerNorm forward / backward
    gate = 3             # gate_concat fwd, gate_concat bwd, gate_finish
    return 2 * (fwd_mod + bwd_mod) + pair + gate


def kernel_probe(args, dev, clips, C, pk):
    """Time the dominant kernel of the step alone, with CUDA events on the launching stream -> roofline object.
    Dominant kernel per the ncu launch list under profiles/: ln_bwd_tma_kernel<2>, the fused MGFM+MLFM LayerNorm /
    BatchNorm backward (HBM-bound: reads dZ, U_g, X_g, U_l, X_l; writes dV_g, dV_l = 7 bf16 passes over [rows, C])."""
    import ctypes as Ct
    from glfusion_b200 import _lib as L
    lib = L.load()
    rows = clips * F * V * HH * WW

    def bf(*shape):
        return torch.randn(*shape, device=dev).to(torch.bfloat16)
    U, X = [bf(rows, C), bf(rows, C)], [bf(rows, C), bf(rows, C)]
    dZ = bf(rows, C)
    dV = [torch.empty_like(U[0]), torch.empty_like(U[0])]
    vec = [torch.rand(5, C, device=dev) + 0.5 for _ in range(2)]
    rowst = [torch.rand(2, rows, device=dev) + 0.5 for _ in range(2)]
    part = [torch.empty(lib.glf_bn_res_ln_bwd_max_blocks() * 4 * C, device=dev) for _ in range(2)]
    nb = Ct.c_int(0)
    stream = Ct.c_void_p(torch.cuda.current_stream().cuda_stream)

    def tab(ts):
        return (Ct.c_void_p * 2)(*[t.data_ptr() for t in ts])
    args_ = (rows, C, L.ptr(dZ), tab(U), tab(X), tab([v[0] for v in vec]), tab([v[1] for v in vec]),
             tab([v[3] for v in vec]), tab([v[4] for v in vec]), tab([v[2] for v in vec]),
             tab([t[0] for t in rowst]), tab([t[1] for t in rowst]), tab(dV), tab(part), Ct.byref(nb), stream)

    def launch():
        L.check(lib.glf_bn_res_ln_pair_bwd(*args_))
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 10
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    alg_bytes = 7 * rows * C * 2          # read dZ, U_g, X_g, U_l, X_l ; write dV_g, dV_l  (bf16)
    achieved = alg_bytes / (ms * 1e-3) / 1e9
    traffic = None                        # DRAM bytes per launch from the committed ncu --set full capture
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        t = json.load(open(tp))
        if t.get("rows") == rows and t.get("C") == C and t.get("kernel") == "ln_bwd_tma_kernel<2>":
            traffic = int(t["traffic_bytes"])
    return {"roofline": {"bound": "hbm", "kernel": "ln_bwd_tma_kernel<2>", "achieved": round(achieved, 1),
                         "peak": pk["hbm_gbs"], "peak_source": pk["source"], "unit": "GB/s",
                         "frac": round(achieved / pk["hbm_gbs"], 4), "traffic": traffic,
                         "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": round(ms, 4),
                         "inputs": "7 x 205 MB per launch, larger than the 126 MB L2"}}


def gram_probe(dev, clips, C, pk):
    """The largest tensor-core product of the Gram form, timed alone: S_b = X_b^T X_b per sequence (glf_gramk.cu: one CTA
    per sequence, operands streamed once, fp32 accumulate in TMEM, column sums on the side).  2 N C^2 FLOPs per sequence
    over N C bf16 bytes = 256 FLOP/B at C = 256: above the ridge (1374.6 TFLOP/s / 6.538 TB/s = 210), so the bound is
    the tensor pipe (the HBM time of the same launch is reported beside it)."""
    import ctypes as Ct
    from glfusion_b200 import _lib as L
    lib = L.load()
    B, N = clips * F, V * HH * WW
    X = torch.randn(B, N, C, device=dev).to(torch.bfloat16)
    D = torch.empty(B, C, C, device=dev, dtype=torch.bfloat16)
    rs = torch.empty(B, C, device=dev)
    stream = Ct.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        L.check(lib.glf_gram_contraction(L.ptr(X), L.ptr(X), L.ptr(D), L.ptr(rs), B, N, C, C, stream))
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 10
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    flops = 2.0 * B * N * C * C
    ach = flops / (ms * 1e-3) / 1e12
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tp):
        t = json.load(open(tp)).get("secondary", {})
        if t.get("rows") == B * N and t.get("C") == C and t.get("kernel") == "gram_kernel":
            traffic = int(t["traffic_bytes"])
    return {"bound": "tensor", "kernel": "gram_kernel (S = X^T X per sequence, + column sums)",
            "achieved": round(ach, 1), "peak": pk["bf16_tflops_burst"],
            "peak_source": pk["source"] + " (burst figure: the kernel is timed alone)", "unit": "TFLOP/s",
            "frac": round(ach / pk["bf16_tflops_burst"], 4), "frac_of_sustained": round(ach / pk["bf16_tflops"], 4),
            "traffic": traffic,
            "algorithmic_flops_per_launch": flops, "ms_per_launch": round(ms, 4),
            "hbm_gbs_same_launch": round(B * N * C * 2 / (ms * 1e-3) / 1e9, 1)}


def gram_family_probe(dev, clips, C, pk, ms_s):
    """gram_kernel as a kernel NAME: per step it runs twice as S = X^T X (1P, glf_gramk.cu symmetric form, timed by
    gram_probe) and twice as R = dV^T X (2P: two inputs, HBM-bound).  R is timed here; the family entry is the four
    launches together against the HBM peak (6P of algorithmic bytes)."""
    import ctypes as Ct
    from glfusion_b200 import _lib as L
    lib = L.load()
    B, N = clips * F, V * HH * WW
    X = torch.randn(B, N, C, device=dev).to(torch.bfloat16)
    dV = torch.randn(B, N, C, device=dev).to(torch.bfloat16)
    D = torch.empty(B, C, C, device=dev, dtype=torch.bfloat16)
    rs = torch.empty(B, C, device=dev)
    stream = Ct.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        L.check(lib.glf_gram_contraction(L.ptr(dV), L.ptr(X), L.ptr(D), L.ptr(rs), B, N, C, C, stream))
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 10
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms_r = e0.elapsed_time(e1) / n
    P = B * N * C * 2
    tot_ms = 2 * ms_s + 2 * ms_r
    ach = 6 * P / (tot_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": "gram_kernel (per step: 2 x S = X^T X, 1P each; 2 x R = dV^T X, 2P each)",
            "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "peak_source": pk["source"], "unit": "GB/s",
            "frac": round(ach / pk["hbm_gbs"], 4), "traffic": None, "algorithmic_bytes_per_launch": int(1.5 * P),
            "ms_per_launch": round(tot_ms / 4, 4), "launches_per_step": 4,
            "ms_S": round(ms_s, 4), "ms_R": round(ms_r, 4),
            "frac_R": round(2 * P / (ms_r * 1e-3) / 1e9 / pk["hbm_gbs"], 4),
            "inputs": "205 MB (S) / 411 MB (R) per launch, larger than the 126 MB L2"}


def dx_gemm_probe(dev, clips, C, pk):
    """The largest tile-GEMM launch of the step, timed alone: dX_b = [dV_b | X_b] [E'_b ; F_b] + e_b (K = 2C, per-sequence
    MN-major B operand, E' = k1 Q + I carries the residual dV; 256 x 256 tiles on CTA pairs, tcgen05.mma.cta_group::2,
    glf_gemm2.cu).  HBM-bound at C = 256: reads dV and X, writes dX = 3 bf16 passes over [rows, C]."""
    import ctypes as Ct
    from glfusion_b200 import _lib as L
    lib = L.load()
    B, N = clips * F, V * HH * WW
    A = torch.randn(B, N, 2 * C, device=dev).to(torch.bfloat16)           # [dV | X] side by side
    Bm = (torch.randn(B, 2 * C, C, device=dev) * 0.05).to(torch.bfloat16)   # [E ; F] per sequence, read MN-major
    bias = torch.randn(C, device=dev)
    D = torch.empty(B, N, C, device=dev, dtype=torch.bfloat16)
    stream = Ct.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        # (no addend: the residual dV is folded into the first operand, E' = E + I, glf_chain.cu)
        L.check(lib.glf_gemm_bf16(L.ptr(A), L.ptr(Bm), L.ptr(D), N, C, 2 * C, B, 0, 1, 2 * C, C, C, N * 2 * C,
                                  C * 2 * C, N * C, L.ptr(bias), 1.0, None, 2 * C, N * 2 * C, 0, 1, None, stream))
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 10
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    alg_bytes = 3 * B * N * C * 2
    ach = alg_bytes / (ms * 1e-3) / 1e9
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    traffic = None
    if os.path.exists(tp):
        t = json.load(open(tp)).get("gemm_dx", {})
        if t.get("rows") == B * N and t.get("C") == C:
            traffic = int(t["traffic_bytes"])
    return {"bound": "hbm", "kernel": "gemm_pair_kernel<A_MN=0, B_MN=1> (dX = [dV | X][E' ; F] + e, K = 2C, cta_group::2)",
            "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "peak_source": pk["source"], "unit": "GB/s",
            "frac": round(ach / pk["hbm_gbs"], 4), "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
            "ms_per_launch": round(ms, 4), "inputs": "617 MB per launch, larger than the 126 MB L2"}


def u_gemm_probe(dev, clips, C, pk):
    """The forward's big product, timed alone: U_b = X_b Q_b^T + c_b (K = C, one [C x C] operand per sequence kept resident
    in shared memory, per-sequence bias, BatchNorm column statistics in the epilogue; glf_gemm3.cu).  HBM-bound: reads X,
    writes U = 2 bf16 passes over [rows, C]."""
    import ctypes as Ct
    from glfusion_b200 import _lib as L
    lib = L.load()
    B, N = clips * F, V * HH * WW
    A = torch.randn(B, N, C, device=dev).to(torch.bfloat16)
    Bm = (torch.randn(B, C, C, device=dev) * 0.05).to(torch.bfloat16)
    bias = torch.randn(C, device=dev)
    D = torch.empty(B, N, C, device=dev, dtype=torch.bfloat16)
    cs = torch.zeros(B * ((N + 127) // 128) * 4, 2, C, device=dev)
    stream = Ct.c_void_p(torch.cuda.current_stream().cuda_stream)

    def launch():
        L.check(lib.glf_gemm_bf16(L.ptr(A), L.ptr(Bm), L.ptr(D), N, C, C, B, 0, 0, C, C, C, N * C, C * C, N * C,
                                  L.ptr(bias), 1.0, None, C, N * C, 0, 1, L.ptr(cs), stream))
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 10
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    alg_bytes = 2 * B * N * C * 2
    ach = alg_bytes / (ms * 1e-3) / 1e9
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    traffic = None
    if os.path.exists(tp):
        t = json.load(open(tp)).get("gemm_u", {})
        if t.get("rows") == B * N and t.get("C") == C:
            traffic = int(t["traffic_bytes"])
    return {"bound": "hbm", "kernel": "gemm_bres_kernel (U = X Q^T + c, K = C, per-sequence B operand resident in shared memory)",
            "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "peak_source": pk["source"], "unit": "GB/s",
            "frac": round(ach / pk["hbm_gbs"], 4), "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
            "ms_per_launch": round(ms, 4), "inputs": "206 MB per launch, larger than the 126 MB L2"}


# ------------------------------------------------------------------------------------------------------------------
def reference_kind() -> str:
    """'reference' when oracle/_ref holds the unmodified reference module (staged by build() from /root/reference),
    else 'port' (the oracle's op-for-op restatement)."""
    from oracle import build_ref
    return "reference" if build_ref.load_reference_tpavi() is not None else "port"


def cpu_step(C: int, clips: int, seed: int = 0):
    """One fwd+bwd of the reference's own fusion path on the host: two UNMODIFIED reference TPAVIModules
    (oracle/_ref/models/TPAVI.py) inside the literal call-site lines R/models/ours.py:1802-1834 (fp32, N x N attention
    materialised, autograd backward); the oracle port of the same algorithm when oracle/_ref was never staged."""
    from oracle import build_ref
    from oracle import tpavi_oracle as O
    B = clips * F
    g = torch.Generator().manual_seed(seed)
    f4 = [torch.randn(B, C, HH, WW, generator=g) for _ in range(V)]
    cl = [torch.randn(B, NCLS, HH, WW, generator=g) for _ in range(V)]
    ct = [torch.randn(B, 1, HH, WW, generator=g) for _ in range(V)]
    do = [torch.randn(B, C, HH, WW, generator=g) for _ in range(V)]
    pg = O.init_params(C, seed=0, randomize_affine=True)
    pl = O.init_params(C, seed=1, randomize_affine=True)
    TPAVI = build_ref.load_reference_tpavi()
    t0 = time.perf_counter()
    if TPAVI is not None:
        build_ref.reference_fusion_fwd_bwd(TPAVI, f4, cl, ct, do, pg, pl)
    else:
        O.fusion_fwd_bwd(f4, cl, ct, do, pg, pl)
    return time.perf_counter() - t0


def width2048(dev, pk, reps: int = 10):
    """Secondary object: the same fused node at the reference NETWORK's own fusion width (R/models/ours.py:1746-1747:
    in_channels = 2048; 3 views x 28 x 28 = 2 352 tokens per frame, N < 5 C -> token-space form), 8 frames, fwd + bwd
    replayed from a CUDA graph.  Tensor-bound: reported against the sustained bf16 tensor peak."""
    C2, V2, B2 = 2048, 3, 8
    f = seeded_fusion(C2, dev)
    g = torch.Generator().manual_seed(5)
    f4 = [torch.randn(B2, C2, HH, WW, generator=g).to(dev).to(torch.bfloat16).requires_grad_(True) for _ in range(V2)]
    cl = [torch.randn(B2, NCLS, HH, WW, generator=g).to(dev) for _ in range(V2)]
    ct = [torch.randn(B2, 1, HH, WW, generator=g).to(dev) for _ in range(V2)]
    dz = torch.randn(B2, V2, HH, WW, C2, generator=g).to(dev).to(torch.bfloat16).permute(0, 4, 1, 2, 3)
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
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    rows = B2 * V2 * HH * WW
    flops = 2 * 13.5 * rows * C2 * C2      # token-space form, both blocks, fwd + bwd (DESIGN.md section 2)
    tf = flops / (ms * 1e-3) / 1e12
    return {"workload": "C=2048, 3 views x 28x28 = 2352 tokens per frame, 8 frames, fwd+bwd of the fused node (token-space form)",
            "ms_per_step": round(ms, 4), "frames_per_s": round(B2 / (ms * 1e-3), 1), "clips_per_s": round(B2 / F / (ms * 1e-3), 1),
            "bound": "tensor", "achieved": round(tf, 1), "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
            "frac": round(tf / pk["bf16_tflops"], 4), "frac_of_burst_peak": round(tf / pk["bf16_tflops_burst"], 4),
            "flops_per_step": flops, "timing": f"{reps} CUDA-graph replays after 3 warm-up replays, 2.7 GB working set >> L2"}


def gpu_reference(C: int, dev):
    """The number to beat on the same box (SURVEY section 2.2 / 8d): the UNMODIFIED reference module pair in PyTorch
    eager mode on this GPU, fp32 (as shipped) and under bf16 autocast, one clip (16 sequences) per step."""
    from oracle import build_ref
    from oracle import tpavi_oracle as O
    TPAVI = build_ref.load_reference_tpavi()
    if TPAVI is None:
        return {"unavailable": "oracle/_ref was not staged (no /root/reference at build time)"}
    B = F
    g = torch.Generator().manual_seed(0)
    f4 = [torch.randn(B, C, HH, WW, generator=g).to(dev) for _ in range(V)]
    cl = [torch.randn(B, NCLS, HH, WW, generator=g).to(dev) for _ in range(V)]
    ct = [torch.randn(B, 1, HH, WW, generator=g).to(dev) for _ in range(V)]
    do = [torch.randn(B, C, HH, WW, generator=g).to(dev) for _ in range(V)]
    pg = {k: v.to(dev) for k, v in O.init_params(C, seed=0, randomize_affine=True).items()}
    pl = {k: v.to(dev) for k, v in O.init_params(C, seed=1, randomize_affine=True).items()}
    res = {"unit": "clips/s", "sample": "1 clip (16 sequences x 3136 tokens) per step, unmodified R/models/TPAVI.py x 2 + "
                                        "the call-site lines ours.py:1802-1834, PyTorch eager, CUDA-event timed, best of 5"}
    for name, ac in (("fp32", False), ("bf16_autocast", True)):
        ts = []
        for i in range(7):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
                build_ref.reference_fusion_fwd_bwd(TPAVI, f4, cl, ct, do, pg, pl)
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(e0.elapsed_time(e1))
        res[name] = round(1.0 / (min(ts) * 1e-3), 2)
    return res


def cpu_baseline(C: int, seconds: float = 15.0):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cpu_step(C, 1)                       # warm-up
    times = []
    t_start = time.perf_counter()
    while len(times) < 3 or (time.perf_counter() - t_start < seconds and len(times) < 20):
        times.append(cpu_step(C, 1))
    best = min(times)
    kind = reference_kind()
    what = ("the unmodified reference module pair (oracle/_ref/models/TPAVI.py) in the call-site lines ours.py:1802-1834"
            if kind == "reference" else "the oracle port of the reference algorithm")
    return {"value": round(1.0 / best, 4), "unit": "clips/s", "cores": cores, "kind": kind,
            "sample": f"1 clip (16 sequences x 3136 tokens, C={C}) fp32 fwd+bwd of {what} "
                      f"(N x N attention materialised), best of {len(times)} after 1 warm-up"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    C = args.channels
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    for _ in range(max(args.warmup, 1)):
        cpu_step(C, 1)
    t0 = time.perf_counter()
    steps = max(1, args.steps)
    for _ in range(steps):
        cpu_step(C, 1)
    dt = (time.perf_counter() - t0) / steps
    val = round(1.0 / dt, 4)
    out = {
        "impl": "reference", "metric": "fusion fwd+bwd clips/sec", "value": val, "unit": "clips/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": steps, "warmup": max(args.warmup, 1),
        "ms_per_step": round(dt * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE configs[1]: MGFM+MLFM modules only, 4 views x 16 frames x 28x28 tokens, C={C}, "
                               "fwd+bwd, frames-as-batch; bounded sample: 1 clip per step on the host CPU"},
        "cpu_baseline": {"value": val, "unit": "clips/s", "cores": cores, "kind": reference_kind(),
                         "sample": "1 clip per step, " + ("the unmodified reference module pair (oracle/_ref/models/TPAVI.py)"
                                                          if reference_kind() == "reference" else
                                                          "oracle port of the reference algorithm") +
                                   " in the call-site lines ours.py:1802-1834 (fp32, N x N materialised)"},
        "e2e": {"value": val, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(out)


_JSON_FD = None


def _claim_stdout():
    """Keep fd 1 for the ONE JSON line: anything libraries print to stdout (e.g. NCCL's version banner) goes to
    stderr instead."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def log(msg: str) -> None:
    """Diagnostics go to stderr: stdout carries only the JSON line."""
    sys.stderr.write(msg + "\n")
    sys.stderr.flush()


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips", type=int, default=8, help="clips per GPU per step")
    ap.add_argument("--channels", type=int, default=256)
    ap.add_argument("--graph", type=int, default=1, help="replay the step from a CUDA graph")
    ap.add_argument("--settle-ms", type=float, default=300.0,
                    help="untimed load before the timed region (steady-state clocks); 0 = time the cold burst only")
    ap.add_argument("--p2p-allreduce", type=int, default=1, help="gradient all-reduce as one NVLink peer-memory kernel")
    ap.add_argument("--graph-allreduce", type=int, default=-1, help="capture the NCCL gradient all-reduce in the step graph")
    ap.add_argument("--overlap-allreduce", type=int, default=1,
                    help="start the peer-memory all-reduce as soon as the weight gradients are final (beside the gate backward)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-width2048", action="store_true", help="skip the C=2048 secondary object")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's output and gradients to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
