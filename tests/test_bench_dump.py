"""CPU: bench.py --dump-outputs writes float32 .npy files: whole outputs when they fit in DUMP_LIMIT, otherwise the same
fixed, seeded sample of distinct positions of every output, identical from call to call."""
import os

import numpy as np
import torch

import bench


def _outputs(b=3, n=16):
    i = torch.arange(b * n * n, dtype=torch.float32).reshape(b, 1, n, n)   # value = flat position
    return {"intensity": i, "adjoint": torch.complex(i, -2 * i)}           # tied to intensity: shows matching positions


def test_dump_whole_outputs(tmp_path):
    out = _outputs()
    bench.dump_outputs(str(tmp_path), out)
    i, a = np.load(tmp_path / "intensity.npy"), np.load(tmp_path / "adjoint.npy")
    assert i.dtype == a.dtype == np.float32
    assert np.array_equal(i, out["intensity"].numpy())
    assert np.array_equal(a, torch.view_as_real(out["adjoint"]).numpy())


def test_dump_sample_is_fixed_and_within_the_limit(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT", 2 * 1024 + 12 * 100)        # 100 positions of 4 + 8 bytes
    out = _outputs()
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), out)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= bench.DUMP_LIMIT
    i, a = np.load(tmp_path / "a" / "intensity.npy"), np.load(tmp_path / "a" / "adjoint.npy")
    assert i.dtype == a.dtype == np.float32 and i.shape == (100,) and a.shape == (100, 2)
    assert np.all(np.diff(i) > 0) and i[0] >= 0 and i[-1] < 3 * 16 * 16     # distinct positions, in order
    assert len(np.unique(i // (3 * 16 * 16 / 100))) > 90                       # spread over the whole output
    assert np.array_equal(a[:, 0], i) and np.array_equal(a[:, 1], -2 * i)
    for f in ("intensity.npy", "adjoint.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
