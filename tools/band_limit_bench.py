"""Cost of the band-limit option on one GPU.  Every config is timed three ways:
  (a) the plain entry point (asm_b200_forward / _adjoint / _focal_stack),
  (b) its _bl entry point with band_limit = 0 (must cost the same as (a): the same launches),
  (c) its _bl entry point with band_limit = 1.
CUDA events, warm-up first, the three ways interleaved over --rounds rounds (the spread of the rounds is the run-to-run
spread); the inputs of a timed window rotate over enough copies to exceed 256 MB.  Writes one JSON file into --out, with
the card's name, power limit and SM clocks read in the same run.

    python tools/band_limit_bench.py --out DIR [--steps 20] [--warmup 3] [--rounds 3]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from focus_bench import card, timed  # noqa: E402

LAMB, PX = 532e-9, 1.5e-6
ROTATE_BYTES = 256 << 20
# (name, N, zero_padding, B, adjoint too, z_max; K for a focal stack)
CONFIGS = [dict(name="c2", n=256, pad=False, b=4096, adjoint=False, z_max=1e-3),
           dict(name="c3", n=1024, pad=False, b=512, adjoint=True, z_max=6e-3),
           dict(name="c3pad", n=1024, pad=True, b=512, adjoint=True, z_max=6e-3),
           dict(name="focal_c3_like", n=1024, pad=False, b=16, k=16, z_max=6e-3)]


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def run_config(L, cfg, steps, warmup, rounds):
    lib = L.load()
    dev = torch.device("cuda:0")
    n, b, pad = cfg["n"], cfg["b"], cfg["pad"]
    k = cfg.get("k")
    rng = np.random.default_rng(0)
    per_copy = b * n * n * 8
    copies = max(1, -(-ROTATE_BYTES // per_copy))
    xs = [torch.from_numpy((rng.standard_normal((b, 1, n, n)) + 1j * rng.standard_normal((b, 1, n, n)))
                           .astype(np.complex64)).to(dev) for _ in range(copies)]
    z = torch.from_numpy(rng.uniform(0.1 * cfg["z_max"], cfg["z_max"], (b, k) if k else b).astype(np.float32)).to(dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    if k:
        need = lib.asm_b200_focal_stack_workspace_bytes(b, k, n, int(pad))
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        out = torch.empty((b, k, n, n), dtype=torch.float32, device=dev)

        def call(flag):
            def step(x):
                args = (_p(x), None, _p(z), L.Z_F32, k, _p(out), None, None, b, n, int(pad), L.IN_COMPLEX,
                        L.OUT_INTENSITY, LAMB, PX, 1.0, _p(ws), need, st)
                L.check(lib.asm_b200_focal_stack(*args) if flag is None else lib.asm_b200_focal_stack_bl(*args, flag))
            return step
        units = b * k
    else:
        need = lib.asm_b200_workspace_bytes(b, 1, n, int(pad))
        ws = torch.empty(need, dtype=torch.uint8, device=dev)
        out = torch.empty((b, 1, n, n), dtype=torch.complex64, device=dev)
        out_a = torch.empty_like(out) if cfg["adjoint"] else None

        def call(flag):
            def step(x):
                fa = (_p(x), None, _p(z), L.Z_F32, _p(out), None, b, 1, n, int(pad), L.IN_COMPLEX, L.OUT_COMPLEX,
                      LAMB, PX, 1.0, 1.0, _p(ws), need, st)
                L.check(lib.asm_b200_forward(*fa) if flag is None else lib.asm_b200_forward_bl(*fa, flag))
                if out_a is not None:
                    aa = (_p(x), None, _p(z), L.Z_F32, None, None, _p(out_a), None, b, 1, n, int(pad), L.IN_COMPLEX,
                          L.OUT_COMPLEX, LAMB, PX, 1.0, _p(ws), need, st)
                    L.check(lib.asm_b200_adjoint(*aa) if flag is None else lib.asm_b200_adjoint_bl(*aa, flag))
            return step
        units = b
    ways = {"a_plain": None, "b_bl0": 0, "c_bl1": 1}
    ms = {w: [] for w in ways}
    for _ in range(rounds):
        for w, flag in ways.items():
            ms[w].append(timed(call(flag), xs, steps, warmup))
    res = {"config": cfg, "rotated_bytes": copies * per_copy, "units_per_step": units}
    for w in ways:
        v = np.array(ms[w])
        res[w] = {"ms_per_step": v.tolist(), "median_ms": float(np.median(v)),
                  "spread_pct": float(100 * (v.max() - v.min()) / np.median(v)),
                  "units_per_s": float(units / (np.median(v) * 1e-3))}
    base = res["a_plain"]["median_ms"]
    res["b_vs_a_pct"] = 100 * (res["b_bl0"]["median_ms"] / base - 1)
    res["c_vs_a_pct"] = 100 * (res["c_bl1"]["median_ms"] / base - 1)
    print(json.dumps({"name": cfg["name"], **{w: round(res[w]["median_ms"], 3) for w in ways},
                      "spread_pct": round(res["a_plain"]["spread_pct"], 2), "b_vs_a_pct": round(res["b_vs_a_pct"], 2),
                      "c_vs_a_pct": round(res["c_vs_a_pct"], 2)}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("band_limit_bench needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as pkg
    L = pkg._lib
    results = {"card": card(), "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
               "configs": [run_config(L, cfg, a.steps, a.warmup, a.rounds) for cfg in CONFIGS],
               "card_after": card()}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "band_limit_bench.json"), "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
