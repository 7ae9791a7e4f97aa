"""GPU: bench.py prints ONE JSON line with every key of the measurement contract (value / e2e / roofline /
cpu_baseline / clocks / gpu_launches), for our arm and for the reference (CPU) arm."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_bench_line_ours():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    d = _run("--steps", "3", "--warmup", "3", "--batch", "64", "--e2e-batch", "16", "--ref-cuda-units", "8")
    assert d["metric"].startswith("ASM holograms/s") and d["unit"] == "units/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["value"] > 1000 and abs(d["value"] - 64 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12
    assert abs(rf["achieved"] - d["value"] * 28 * 1024 * 1024 / 1e9) < 1e-6 * rf["achieved"]
    assert d["gpu_launches"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    p = d["parity"]
    assert p["ok"] and p["intensity"] < 1e-4 and p["adjoint"] < 1e-4      # the timed outputs, against the float64 oracle
    gb = d["gpu_torch_baseline"]
    assert gb["value"] > 0 and gb["speedup_device_resident"] > 1.0       # the reference's torch.fft path on the same GPU
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs writes what the last timed step computed; 4 units at 1024^2 fit in 64 MB, so the whole batch is
    written.  The last unit, which the parity spot check does not look at, against the float64 oracle."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import numpy as np
    import bench
    from oracle import asm_oracle as ao
    d = _run("--steps", "2", "--warmup", "3", "--batch", "4", "--no-e2e", "--no-cpu", "--no-gpu-baseline",
             "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    i, a = np.load(tmp_path / "intensity.npy"), np.load(tmp_path / "adjoint.npy")
    assert i.dtype == a.dtype == np.float32 and i.shape == (4, 1, 1024, 1024) and a.shape == (4, 1, 1024, 1024, 2)
    O, G, z = bench.synth(bench.CONFIGS["c3"], 4, torch.device("cuda"), 1234)
    o, g, zz = O[3:].cpu().numpy(), G[3:].cpu().numpy(), z[3:].cpu().numpy()
    assert ao.rel_l2(i[3:], np.abs(ao.asm(o, bench.LAMB, zz, bench.PX)) ** 2) < 1e-4
    assert ao.rel_l2(a[3:, ..., 0] + 1j * a[3:, ..., 1], ao.asm_adjoint(g, bench.LAMB, zz, bench.PX)) < 1e-4


def test_bench_line_reference_arm():
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert d["impl"] == "reference" and d["unit"] == "units/s" and d["value"] > 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["value"] == d["value"]


@pytest.mark.parametrize("config,units", [("c2", 4096), ("c3pad", 8), ("c4", 8)])
def test_bench_other_configs(config, units):
    """--config switches the workload (BASELINE.json configs[1], configs[2] padded, configs[3]); strong scaling keeps the
    global batch fixed."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    d = _run("--config", config, "--steps", "2", "--warmup", "3", "--batch", str(units), "--no-e2e", "--no-cpu",
             "--no-gpu-baseline", "--scaling", "strong")
    assert d["config"]["name"] == config and d["scaling"] == "strong" and d["config"]["global_batch"] == units
    n = d["config"]["n"]
    bpu = (28 if config != "c2" else 12) * n * n
    assert d["roofline"]["bytes_per_unit"] == bpu
    assert abs(d["roofline"]["achieved"] - d["value"] * bpu / 1e9) < 1e-6 * d["roofline"]["achieved"]
    assert d["parity"]["ok"]
