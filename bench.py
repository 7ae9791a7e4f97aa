#!/usr/bin/env python
"""bench.py -- ASM holograms/s (fwd+adjoint) @1024^2 on B200 (BASELINE.json metric) and the other named configs.

A step = one pass of the hot path over one batch of synthetic fields: B forward propagations (complex64 field ->
fp32 |U|^2) plus, for the fwd+adjoint configs, B adjoint propagations (complex64 cotangent -> complex64).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c3]   our CUDA path (default c3 = the headline)
  python bench.py --impl reference ...        the reference's own torch code on the host CPU cores
  python bench.py --impl reference-cuda ...   the reference's own torch code (cuFFT) on the same GPU
  python bench.py ... --dump-outputs DIR      also write what the last timed step computed as DIR/*.npy
                                              (rank 0's batch only: with N > 1 GPUs a shard, or one of N batches,
                                              so compare dumps taken with the same --gpus)

  --config  c2    256^2  forward only, B = 4096               (BASELINE.json configs[1])
            c3    1024^2 fwd+adjoint,  B = 512, unpadded      (configs[2], the metric's config; default)
            c3pad 1024^2 fwd+adjoint,  B = 512, zero_padding=True (FFT 2048; what Holo_Generator calls, Forward_model.py:24)
            c4    2048^2 fwd+adjoint,  B = 128, unpadded      (configs[3])
            c4pad 2048^2 fwd+adjoint,  B = 128, zero_padding=True (FFT 4096)
  --scaling weak (default: B samples per GPU) | strong (B samples in total, contiguous shards per rank)

Prints ONE JSON line (rank 0).  `value` is device-resident throughput; `e2e` goes through the drop-in Python API
(`ASM(...)`, utils/Angular_Spectrum_Method.py:7) with pinned HOST buffers (H2D of the inputs and D2H of the results
inside the timed region); `parity` is a spot check of the timed step's outputs against the float64 oracle.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LAMB, PX = 532e-9, 1.5e-6
DUMP_LIMIT = 64 * 10**6          # bytes written by --dump-outputs in all
CONFIGS = {
    # name: field size, batch, padding, adjoint leg, z_max [m], CPU-arm sample (units per step), BASELINE.json config
    "c2": dict(n=256, batch=4096, pad=False, adjoint=False, z_max=1e-3, cpu_units=64,
               label="configs[1]: synthetic batched ASM forward 256x256 complex64, batch 4096, random per-sample z"),
    "c3": dict(n=1024, batch=512, pad=False, adjoint=True, z_max=6e-3, cpu_units=4,
               label="configs[2]: synthetic ASM fwd+adjoint 1024x1024 complex64, unpadded (M = N)"),
    "c3pad": dict(n=1024, batch=512, pad=True, adjoint=True, z_max=6e-3, cpu_units=2,
                  label="configs[2] with zero_padding=True (FFT 2048): ASM fwd+adjoint 1024x1024 complex64"),
    "c4": dict(n=2048, batch=128, pad=False, adjoint=True, z_max=6e-3, cpu_units=2,
               label="configs[3]: synthetic ASM fwd+adjoint 2048x2048 complex64, unpadded (M = N)"),
    "c4pad": dict(n=2048, batch=128, pad=True, adjoint=True, z_max=6e-3, cpu_units=1,
                  label="configs[3] with zero_padding=True (FFT 4096): ASM fwd+adjoint 2048x2048 complex64"),
}


def bytes_per_unit(cfg) -> int:
    """SURVEY.md 8(d): forward 12 N^2 (complex64 in, fp32 out), adjoint 16 N^2; counted on the N x N field."""
    return (12 + (16 if cfg["adjoint"] else 0)) * cfg["n"] * cfg["n"]


def metric_name(cfg) -> str:
    n = cfg["n"]
    return f"ASM holograms/s ({'fwd+adjoint' if cfg['adjoint'] else 'forward'}) @{n}^2"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic(config: str):
    """DRAM bytes per unit measured with ncu for the committed build (profiles/r02_dram_traffic.json, written by
    tools/dram_traffic.py); None when no capture exists for this config."""
    p = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    try:
        rec = json.load(open(p))["configs"][config]
        return float(rec["dram_bytes_per_unit"]), f"profiles/r02_dram_traffic.json ({rec.get('how', 'ncu')})"
    except Exception:
        return None, None


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (NVML every 5 ms; nvidia-smi as a fallback)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thr, self.stop_flag, self.nvml = index, [], None, None, False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.thr = threading.Thread(target=self._poll, daemon=True)
            self.thr.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thr = threading.Thread(target=self._read, daemon=True)
        self.thr.start()

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((time.time(), mhz, mask))
            except Exception:
                pass
            time.sleep(0.005)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.nvml is not None:
            self.stop_flag = True
            self.thr.join(timeout=1.0)
            rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows
            sm = [r[1] for r in rows]
            reasons = sorted({name for r in rows for (name, bit) in self.REASONS if r[2] & bit})
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.mx, "reasons": reasons,
                    "samples": len(sm), "source": "nvml, 5 ms period, inside the timed region"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 and len(r) >= 7] or [r for (_, r) in self.rows if len(r) >= 7]
        sm, mx, reasons = [], None, set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi -lms 20"}


def bind_to_gpu_numa_node(local_rank: int) -> str:
    """Pin this process (and therefore its pinned host buffers, first-touch) to the CPUs next to its GPU.
    Returns a short description for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0"
        cpulist = open(os.path.join(path, "local_cpulist")).read().strip()
        node = open(os.path.join(path, "numa_node")).read().strip()
        cpus = set()
        for part in cpulist.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        allowed = os.sched_getaffinity(0)
        bind_to_gpu_numa_node.original = allowed
        cpus &= allowed
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"numa node {node}, {len(cpus)} cpus"
        return f"numa node {node} (no allowed cpus there; affinity unchanged)"
    except Exception as e:  # no sysfs / no permission: keep the default placement
        return f"unbound ({type(e).__name__})"


# ---------------------------------------------------------------------------------------------------
# reference arms: the reference's own torch code (staged under baseline/_ref by build(), else the oracle's port)
# ---------------------------------------------------------------------------------------------------
def reference_ops():
    """(forward_intensity, adjoint, kind): the reference's ASM + |.|^2 (utils/Forward_model.py:39); the adjoint is
    ASM(g, -z) unpadded (exact) and autograd's VJP through the reference's own graph when padded."""
    import torch
    from oracle import ref_import, torch_port
    if ref_import.available():
        ASM = ref_import.load()[0]
        kind = "reference"
    else:
        def ASM(O, lamb, d, px, requires_grad=True, zero_padding=False):
            return torch_port.asm_torch(O, lamb, d, px, zero_padding)
        kind = "port"

    def fwd(O, z, pad):
        with torch.no_grad():
            return torch.pow(torch.abs(ASM(O, LAMB, z, PX, zero_padding=pad)), 2).float()

    def adj(G, O, z, pad):
        if not pad:
            with torch.no_grad():
                return ASM(G, LAMB, -z, PX)
        x = O.clone().requires_grad_(True)
        U = ASM(x, LAMB, z, PX, zero_padding=True)
        return torch.autograd.grad(U, x, grad_outputs=G.to(U.dtype))[0]

    return fwd, adj, kind


def synth(cfg, units, device, seed):
    import torch
    n = cfg["n"]
    g = torch.Generator(device=device).manual_seed(seed)
    O = torch.polar(0.5 + 0.5 * torch.rand(units, 1, n, n, device=device, generator=g),
                    2 * torch.pi * torch.rand(units, 1, n, n, device=device, generator=g))          # complex64 field
    G = torch.view_as_complex(torch.randn(units, 1, n, n, 2, device=device, generator=g))            # complex64 cotangent
    z = ((0.2 + 0.8 * torch.rand(units, 1, 1, 1, device=device, generator=g)) * cfg["z_max"]).float()
    return O, G, z


def dump_outputs(out_dir, arrays, seed=0):
    """--dump-outputs: write each tensor as out_dir/<name>.npy in float32, complex ones with a trailing (re, im) axis.
    The tensors share one shape.  When they would take more than DUMP_LIMIT bytes together, each is cut down to the same
    fixed sample of k distinct flat positions, in increasing order: one position in each of k equal slices of the flat
    range, drawn by a CPU generator seeded with `seed`.  Equal inputs give identical files from run to run and from
    build to build."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    numel = next(iter(arrays.values())).numel()
    assert all(t.numel() == numel for t in arrays.values())
    per_pos = sum(8 if t.is_complex() else 4 for t in arrays.values())
    budget = DUMP_LIMIT - 1024 * len(arrays)                 # room for the .npy headers
    idx = None
    if numel * per_pos > budget:
        k = budget // per_pos
        lo = (torch.arange(k + 1, dtype=torch.float64) * (numel / k)).long()       # slice bounds, lo[k] == numel
        width = lo[1:] - lo[:-1]                                                    # >= 1 because k < numel
        off = (torch.rand(k, generator=torch.Generator().manual_seed(seed), dtype=torch.float64) * width).long()
        idx = lo[:-1] + torch.minimum(off, width - 1)
    for name, t in arrays.items():
        x = t if idx is None else t.reshape(-1)[idx.to(t.device)]
        x = torch.view_as_real(x) if x.is_complex() else x
        np.save(os.path.join(out_dir, f"{name}.npy"), x.float().cpu().numpy())


def cpu_units_per_s(cfg, repeats: int, warmup: int):
    import torch
    orig = getattr(bind_to_gpu_numa_node, "original", None)
    if orig:                                       # the CPU arm uses every host core, not only the GPU's NUMA node
        os.sched_setaffinity(0, orig)
    torch.set_num_threads(len(os.sched_getaffinity(0)) or 1)
    fwd, adj, kind = reference_ops()
    units = cfg["cpu_units"]
    O, G, z = synth(cfg, units, torch.device("cpu"), 1234)
    times = []
    for i in range(warmup + repeats):
        t0 = time.perf_counter()
        fwd(O, z, cfg["pad"])
        if cfg["adjoint"]:
            adj(G, O, z, cfg["pad"])
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return times, torch.get_num_threads(), kind, units


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, threads, kind, units = cpu_units_per_s(cfg, max(1, args.steps), args.warmup)
    total = sum(times)
    v = units * len(times) / total
    line = {"impl": "reference", "metric": metric_name(cfg), "value": v, "unit": "units/s",
            "n_gpus": args.gpus, "steps": len(times), "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32 (complex64 fft / complex128 ifft)", "data": "synthetic",
            "config": {"workload": f"{cfg['label']}; each step = {units} units on the host CPU", "name": args.config,
                       "n": cfg["n"], "zero_padding": cfg["pad"]},
            "cpu_baseline": {"value": v, "unit": "units/s", "cores": threads, "kind": kind,
                             "sample": f"{units} units per step x {len(times)} steps, torch CPU, "
                                       + ("the reference's own utils/Angular_Spectrum_Method.py (staged in baseline/_ref)"
                                          if kind == "reference" else "oracle/torch_port.py")},
            "e2e": {"value": v, "unit": "units/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def torch_cuda_units_per_s(cfg, dev, steps: int, warmup: int, units_total: int):
    """The reference's torch code on the SAME GPU (cuFFT + ~12 elementwise launches, complex128 temporaries), chunked
    so that its B x M x M complex128 temporaries fit; CUDA-event timing."""
    import torch
    fwd, adj, kind = reference_ops()
    m = cfg["n"] * (2 if cfg["pad"] else 1)
    chunk = max(1, min(units_total, (1 << 28) // (m * m)))            # <= 256 Mi pixels of complex128 temporaries per op
    O, G, z = synth(cfg, units_total, dev, 1234)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step():
        for s in range(0, units_total, chunk):
            fwd(O[s:s + chunk], z[s:s + chunk], cfg["pad"])
            if cfg["adjoint"]:
                adj(G[s:s + chunk], O[s:s + chunk], z[s:s + chunk], cfg["pad"])

    for _ in range(max(1, warmup)):
        step()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    return units_total / (ms * 1e-3), ms, kind, chunk


def run_reference_cuda(args, cfg):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    units = min(cfg["batch"], args.ref_cuda_units)
    v, ms, kind, chunk = torch_cuda_units_per_s(cfg, dev, max(1, args.steps), args.warmup, units)
    line = {"impl": "reference-cuda", "metric": metric_name(cfg), "value": v, "unit": "units/s", "n_gpus": 1,
            "steps": max(1, args.steps), "warmup": max(1, args.warmup), "ms_per_step": ms, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32 (complex64 cuFFT / complex128 inverse)",
            "data": "synthetic",
            "config": {"workload": f"{cfg['label']}; {units} units per step in chunks of {chunk}, the reference's torch "
                                   f"path on the same B200 ({kind})", "name": args.config, "n": cfg["n"],
                       "zero_padding": cfg["pad"]}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args, cfg):
    import torch
    import torch.distributed as dist
    import style_transfer_based_holographic_imaging_b200 as pkg
    from style_transfer_based_holographic_imaging_b200 import _lib as L
    from style_transfer_based_holographic_imaging_b200.parallel import shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)            # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = L.load()

    n, pad, with_adj = cfg["n"], cfg["pad"], cfg["adjoint"]
    gb = args.batch if args.batch > 0 else cfg["batch"]
    if args.scaling == "strong":
        lo, hi = shard_bounds(gb, rank, world)     # global batch fixed, contiguous shard per rank, no collective
        B, total_units = hi - lo, gb
    else:
        B, total_units = gb, gb * world
    O, G, z = synth(cfg, B, dev, 1234 + rank)
    I = torch.empty(B, 1, n, n, device=dev, dtype=torch.float32)
    A = torch.empty(B, 1, n, n, device=dev, dtype=torch.complex64) if with_adj else None

    def step():
        pkg.asm_forward_raw(O, z, LAMB, PX, pad, out_mode=L.OUT_INTENSITY, out=I)
        if with_adj:
            pkg.asm_adjoint_raw(G, z, LAMB, PX, pad, out=A)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    n0 = lib.asm_b200_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    t1 = time.time()
    launches = lib.asm_b200_launch_count() - n0
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    value = total_units * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:            # I and A still hold what the last timed step wrote
        dump_outputs(args.dump_outputs, {"intensity": I, "adjoint": A} if with_adj else {"intensity": I})

    # ---- parity spot check of what was just timed: 2 samples of I (and A) against the float64 oracle ----
    parity = None
    if rank == 0 and not args.no_parity:
        import numpy as np
        from oracle import asm_oracle as ao
        idx = sorted({min(1, B - 1), max(0, B - 2)})
        o, zz = O[idx].cpu().numpy(), z[idx].cpu().numpy()
        parity = {"samples": idx, "tolerance": 1e-4,
                  "intensity": ao.rel_l2(I[idx].cpu().numpy(), np.abs(ao.asm(o, LAMB, zz, PX, pad)) ** 2)}
        if with_adj:
            parity["adjoint"] = ao.rel_l2(A[idx].cpu().numpy(), ao.asm_adjoint(G[idx].cpu().numpy(), LAMB, zz, PX, pad))
        parity["ok"] = all(v < 1e-4 for k, v in parity.items() if k in ("intensity", "adjoint"))

    # ---- per-pass share of the step (CUDA events inside the library, separate un-timed pass) ----
    lib.asm_b200_profile(1, None)
    step()
    torch.cuda.synchronize()
    ms3 = (ctypes.c_double * 3)()
    lib.asm_b200_profile(0, ms3)
    pass_ms = {"rows_fwd": ms3[0], "cols": ms3[1], "rows_inv": ms3[2]}

    # ---- end to end through the drop-in API (ASM, utils/Angular_Spectrum_Method.py:7) with pinned host buffers ----
    e2e = None
    if not args.no_e2e:
        # whole batch on one GPU; with several ranks on one host the pinned buffers (28 MB per unit) are capped at ~30 GB in total
        Be = min(B, args.e2e_batch) if args.e2e_batch > 0 else (B if world == 1 else max(1, min(B, 1024 // world)))
        chunk = max(1, min(args.e2e_chunk, Be))
        hO = torch.empty(Be, 1, n, n, dtype=torch.complex64, pin_memory=True)
        hI = torch.empty(Be, 1, n, n, dtype=torch.float32, pin_memory=True)
        hO.copy_(O[:Be])
        hz = z[:Be].cpu().pin_memory()
        if with_adj:
            hG = torch.empty(Be, 1, n, n, dtype=torch.complex64, pin_memory=True)
            hA = torch.empty(Be, 1, n, n, dtype=torch.complex64, pin_memory=True)
            hG.copy_(G[:Be])
        streams = [torch.cuda.Stream(device=dev) for _ in range(args.e2e_streams)]

        @torch.no_grad()
        def e2e_step():
            # chunks round-robin over the streams: H2D -> drop-in ASM(...) -> D2H; copies of one chunk overlap the
            # opposite-direction copies and the compute of the others (PCIe is full duplex)
            for ci, s0 in enumerate(range(0, Be, chunk)):
                st = streams[ci % len(streams)]
                with torch.cuda.stream(st):
                    o = hO[s0:s0 + chunk].to(dev, non_blocking=True)
                    zz = hz[s0:s0 + chunk].to(dev, non_blocking=True)
                    U = pkg.ASM(o, LAMB, zz, PX, zero_padding=pad)                       # the reference's call signature
                    hI[s0:s0 + chunk].copy_(torch.pow(torch.abs(U), 2).float(), non_blocking=True)   # Forward_model.py:39
                    if with_adj:
                        gg = hG[s0:s0 + chunk].to(dev, non_blocking=True)
                        if pad:
                            adj = pkg.asm_adjoint_raw(gg, zz, LAMB, PX, True)            # VJP of the padded operator
                        else:
                            adj = pkg.ASM(gg, LAMB, -zz, PX)                             # unpadded adjoint = ASM(g, -z)
                        hA[s0:s0 + chunk].copy_(adj, non_blocking=True)
            for st in streams:
                st.synchronize()

        e2e_step()
        barrier()
        te = time.perf_counter()
        ke = max(1, min(args.steps, 3))
        for _ in range(ke):
            e2e_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - te], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        units_e = torch.tensor([float(Be)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(units_e, op=dist.ReduceOp.SUM)
        h2d = Be * (n * n * 8 * (2 if with_adj else 1) + 4)
        d2h = Be * (n * n * 4 + (n * n * 8 if with_adj else 0))
        e2e = {"value": float(units_e.item()) * ke / dt, "unit": "units/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "h2d_gbs_per_gpu": h2d * ke / dt / 1e9, "d2h_gbs_per_gpu": d2h * ke / dt / 1e9,
               "batch_per_gpu": Be, "steps": ke, "host_binding": numa,
               "api": "style_transfer_based_holographic_imaging_b200.ASM(O, lamb, d, px, zero_padding) + |U|^2 (Forward_model.py:39)",
               "note": f"pinned host buffers, {len(streams)}-stream pipeline over chunks of {chunk}, host wall clock, max over ranks"}

    if rank == 0:
        peak, peak_src = peaks()
        bpu = bytes_per_unit(cfg)
        achieved = value / world * bpu / 1e9          # per-GPU algorithmic GB/s
        traffic_pu, traffic_src = measured_traffic(args.config)
        m = n * (2 if pad else 1)
        calls = 2 if with_adj else 1
        line = {"metric": metric_name(cfg), "value": value, "unit": "units/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": cfg["label"], "name": args.config, "n": n, "fft_size": m, "batch_per_gpu": B,
                           "global_batch": total_units, "zero_padding": pad, "z_max_m": cfg["z_max"],
                           "wavelength": LAMB, "pixel_size": PX,
                           "parallelism": f"batch-sharded x{world}, no collective",
                           "l2": f"inputs {B * n * n * (16 if with_adj else 8) / 2**30:.2f} GiB per step >> 126 MB L2 (no flush needed)"},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": None if traffic_pu is None else traffic_pu * B,
                             "traffic_source": traffic_src, "peak_source": peak_src,
                             "bytes_per_unit": bpu,
                             "kernel": f"whole step = {calls} call(s) x (setup + chunks x {{row FFT, column FFT.H.IFFT, row IFFT}}); "
                                       f"no single kernel owns the HBM traffic, so `achieved` is the step's algorithmic bytes "
                                       f"({bpu} B per unit) over the CUDA-event time of the timed steps",
                             "pass_ms_profiled": pass_ms},
                "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "parity": parity}
        if not args.no_cpu:
            times, threads, kind, units = cpu_units_per_s(cfg, 2, 1)
            line["cpu_baseline"] = {"value": units * len(times) / sum(times), "unit": "units/s", "cores": threads, "kind": kind,
                                    "sample": f"{units} units x {len(times)} repeats after 1 warm-up, torch CPU, "
                                              + ("the reference's own ASM (baseline/_ref)" if kind == "reference"
                                                 else "oracle/torch_port.py")}
        if not args.no_gpu_baseline:
            torch.cuda.empty_cache()
            units = min(B, args.ref_cuda_units)
            v, gms, kind, chunk = torch_cuda_units_per_s(cfg, dev, 2, 1, units)
            line["gpu_torch_baseline"] = {"value": v, "unit": "units/s", "kind": kind,
                                          "sample": f"{units} units per step in chunks of {chunk}, the reference's torch.fft "
                                                    f"path (cuFFT) on the same B200, CUDA events, 2 steps after 1 warm-up",
                                          "speedup_device_resident": value / world / v}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_bw_test(args):
    """bandwidthTest-style host <-> device measurement on every rank at once: pinned H2D and D2H copies of 1 GiB chunks,
    both directions concurrently on two streams, no compute.  Names the host-side bound of the `e2e` leg at N GPUs."""
    import torch
    import torch.distributed as dist
    world, rank, local = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nbytes = 1 << 30
    h_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    d_in = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_out = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    res = {}
    for name, up, dn in (("h2d_only", True, False), ("d2h_only", False, True), ("both", True, True)):
        for timed in (False, True):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(4 if timed else 1):
                if up:
                    with torch.cuda.stream(s_up):
                        d_in.copy_(h_in, non_blocking=True)
                if dn:
                    with torch.cuda.stream(s_dn):
                        h_out.copy_(d_out, non_blocking=True)
            s_up.synchronize(); s_dn.synchronize()
            dt = time.perf_counter() - t0
        gbs = torch.tensor([4 * nbytes / dt / 1e9], device=dev, dtype=torch.float64)     # per direction
        if world > 1:
            mn, sm = gbs.clone(), gbs.clone()
            dist.all_reduce(mn, op=dist.ReduceOp.MIN); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            res[name] = {"per_gpu_min_gbs": float(mn.item()), "aggregate_gbs_per_direction": float(sm.item())}
        else:
            res[name] = {"per_gpu_min_gbs": float(gbs.item()), "aggregate_gbs_per_direction": float(gbs.item())}
    if rank == 0:
        print(json.dumps({"what": "pinned host <-> device copy bandwidth, all ranks at once (1 GiB x 4 per direction)", "n_gpus": world,
                          "host_binding": numa, "host_cpus": len(os.sched_getaffinity(0)), "result": res}), flush=True)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--config", default="c3", choices=list(CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--batch", type=int, default=0, help="override the config's batch (per GPU when weak, global when strong)")
    ap.add_argument("--e2e-batch", type=int, default=0, help="units per GPU in the e2e leg (0 = the whole batch on one GPU, 1024 / N per GPU on N GPUs)")
    ap.add_argument("--e2e-chunk", type=int, default=8)
    ap.add_argument("--e2e-streams", type=int, default=4)
    ap.add_argument("--ref-cuda-units", type=int, default=64)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--bw-test", action="store_true", help="host <-> device copy bandwidth of all ranks at once (names the e2e bound)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's outputs of the last step as DIR/intensity.npy and, for "
                         "the fwd+adjoint configs, DIR/adjoint.npy (float32, adjoint with a trailing (re, im) axis); "
                         "beyond 64 MB in all, the same fixed, seeded sample of positions of each")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.bw_test):
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        return run_reference(args, cfg)
    if args.impl == "reference-cuda":
        return run_reference_cuda(args, cfg)
    if args.bw_test and (args.gpus == 1 or "RANK" in os.environ):
        return run_bw_test(args)
    if args.gpus > 1 and "RANK" not in os.environ:
        # convenience: re-launch under torchrun when called directly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_ours(args, cfg)


if __name__ == "__main__":
    main()
