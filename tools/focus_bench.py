"""Focal-stack throughput on one GPU: (a) focal_stack with moments only, (b) focal_stack with intensity output, against
(c) what a user can do without it: asm_b200_forward (OUT_INTENSITY) on the input replicated to B K samples (replication
outside the timed window) plus a torch reduction to the same three moments.  CUDA events, warm-up first; the input of a
timed window is rotated over enough copies to exceed the 126 MB L2 (the JSON records the bytes).  Writes one JSON
file into --out, with the card's name, power limit and SM clocks read in the same run.

    python tools/focus_bench.py --out DIR [--steps 20] [--warmup 3]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# (name, N, zero_padding, B, K)
CONFIGS = [("mnist_shape", 128, True, 100, 25), ("c3_like", 1024, False, 16, 16),
           ("holo_generator_shape", 1024, True, 4, 16), ("large", 2048, False, 4, 8)]
L2_BYTES = 126 << 20
LAMB, PX = 532e-9, 1.5e-6


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:  # the measurement stays valid; the JSON says what is missing
        return {"error": str(e), "name": torch.cuda.get_device_name(0)}


def timed(fn, inputs, steps, warmup):
    for i in range(warmup):
        fn(inputs[i % len(inputs)])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(inputs[i % len(inputs)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("focus_bench needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as pkg
    from oracle import asm_oracle as ao
    L = pkg._lib
    dev = torch.device("cuda:0")
    res = {"card_before": card(), "steps": a.steps, "warmup": a.warmup, "configs": []}
    for name, n, pad, b, k in CONFIGS:
        g = torch.Generator(device=dev).manual_seed(0)
        x_bytes = b * n * n * 4
        copies = max(2, -(-2 * L2_BYTES // x_bytes))
        xs = [torch.rand((b, n, n), device=dev, generator=g) + 0.05 for _ in range(copies)]   # holograms
        z = torch.linspace(-1.2e-3, 0.0, k, device=dev, dtype=torch.float32)
        zrep = z.repeat(b).reshape(b * k, 1, 1, 1).contiguous()
        planes = b * k

        def stack_mom(x):
            return pkg.focal_stack(x, z, LAMB, PX, pad, hologram=True, output=None, moments=True)

        def stack_int(x):
            return pkg.focal_stack(x, z, LAMB, PX, pad, hologram=True, output="intensity")

        # baseline: replicated input (outside the timed window), one asm_b200_forward call, torch moments
        reps = [x.reshape(b, 1, n, n).repeat_interleave(k, dim=0).contiguous() for x in xs[:2]]
        ws = torch.empty(L.load().asm_b200_workspace_bytes(planes, 1, n, int(pad)), dtype=torch.uint8, device=dev)
        out = torch.empty((planes, 1, n, n), dtype=torch.float32, device=dev)
        from style_transfer_based_holographic_imaging_b200.functional import _ptr, _stream

        def baseline(xr):
            rc = L.load().asm_b200_forward(_ptr(xr), None, _ptr(zrep), L.Z_F32, _ptr(out), None, planes, 1, n, int(pad),
                                           L.IN_SQRT_REAL, L.OUT_INTENSITY, LAMB, PX, 1.0, 1.0, _ptr(ws), ws.numel(), _stream())
            L.check(rc)
            i = out.reshape(b, k, -1)
            return torch.stack([i.sqrt().sum(-1), i.sum(-1), (i * i).sum(-1)], -1).double()

        t_a = timed(stack_mom, xs, a.steps, a.warmup)
        t_b = timed(stack_int, xs, a.steps, a.warmup)
        t_c = timed(baseline, reps, a.steps, a.warmup)
        # spot check: one plane against the float64 oracle, and the moments against the baseline's
        m = stack_mom(xs[0])
        u = ao.asm(np.sqrt(xs[0][:1].double().cpu().numpy()).reshape(1, 1, n, n).astype(np.complex128), LAMB,
                   z[k // 2:k // 2 + 1].cpu().numpy(), PX, zero_padding=pad)
        img = stack_int(xs[0])[0, k // 2].cpu().numpy()
        err = float(np.linalg.norm(img - np.abs(u[0, 0]) ** 2) / np.linalg.norm(np.abs(u[0, 0]) ** 2))
        mb = baseline(reps[0])
        merr = float(((m - mb).abs() / mb.abs()).max())
        del reps, out, ws
        rec = {"name": name, "N": n, "zero_padding": pad, "B": b, "K": k, "planes": planes,
               "input_bytes_per_window": x_bytes * copies, "input_copies": copies,
               "ms_moments_only": t_a, "ms_intensity": t_b, "ms_baseline": t_c,
               "planes_per_s": {"moments_only": planes / t_a * 1e3, "intensity": planes / t_b * 1e3,
                                "baseline": planes / t_c * 1e3},
               "speedup_moments_only": t_c / t_a, "speedup_intensity": t_c / t_b,
               "oracle_rel_l2_one_plane": err, "moments_max_rel_vs_baseline": merr}
        print(json.dumps(rec), flush=True)
        res["configs"].append(rec)
        del xs
        torch.cuda.empty_cache()
    res["card_after"] = card()
    os.makedirs(a.out, exist_ok=True)
    path = os.path.join(a.out, "focus_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(path)


if __name__ == "__main__":
    main()
