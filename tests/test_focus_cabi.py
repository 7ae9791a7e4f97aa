"""CPU: the focal-stack entry points are exported, size their workspace consistently with the single-call workspace,
and validate their arguments as documented in include/asm_b200.h.  No compute calls here."""
import ctypes

import pytest
import torch

E_NULL, E_SHAPE, E_MODE, E_WORKSPACE, E_OPTICS = -1, -2, -3, -4, -5
LAMB, PX = 532e-9, 1.5e-6


@pytest.fixture(scope="module")
def lib():
    from style_transfer_based_holographic_imaging_b200 import build, _lib
    build.build()
    return _lib.load()


def test_symbols_exported(lib):
    from style_transfer_based_holographic_imaging_b200 import _lib
    for name in ("asm_b200_focal_stack_workspace_bytes", "asm_b200_focal_stack"):
        assert hasattr(lib, name)
        assert name in _lib.SYMBOLS


def test_workspace_bytes(lib):
    fs, single = lib.asm_b200_focal_stack_workspace_bytes, lib.asm_b200_workspace_bytes
    bad_shapes = [(1, 101, 1), (1, 3000, 0), (1, 8, 0), (1, 4096, 1), (1, 16, 0), (0, 128, 0)]
    for b, n, pad in bad_shapes:
        assert single(b, 1, n, pad) == 0
        assert fs(b, 4, n, pad) == 0, (b, n, pad)
    for k in (0, -1):
        assert fs(2, k, 128, 0) == 0
    for b, k, n, pad in [(100, 25, 128, 1), (16, 16, 1024, 0), (4, 16, 1024, 1), (4, 8, 2048, 0), (3, 37, 256, 0),
                         (2, 9, 1024, 0), (1, 3, 4096, 0), (2, 5, 92, 1), (1, 1, 32, 0), (5, 2, 512, 1)]:
        need = fs(b, k, n, pad)
        assert need >= single(b, 1, n, pad) > 0, (b, k, n, pad)


def _call(lib, in_mode=0, out_mode=1, out0=256, out1=None, mom=None, k=4, b=1, n=128, pad=0, lamb=LAMB, px=PX,
          ws=256, ws_bytes=1 << 40, in1=None):
    vp = ctypes.c_void_p
    return lib.asm_b200_focal_stack(vp(256), in1 if in1 is None else vp(in1), vp(256), 0, k,
                                    None if out0 is None else vp(out0), None if out1 is None else vp(out1),
                                    None if mom is None else vp(mom), b, n, pad, in_mode, out_mode, lamb, px, 1.0,
                                    vp(ws), ws_bytes, None)


def test_argument_validation(lib):
    assert _call(lib, out0=None, mom=None) == E_NULL
    assert _call(lib, out_mode=3) == E_MODE                          # OUT_REIM_CAT
    assert _call(lib, out_mode=5) == E_MODE
    assert _call(lib, in_mode=3, in1=256) == E_MODE                  # IN_COT_FIELD
    assert _call(lib, in_mode=9) == E_MODE
    assert _call(lib, out_mode=1, out1=256) == E_MODE                # out1 only with OUT_ABS_ANGLE
    assert _call(lib, k=0) == E_SHAPE
    assert _call(lib, b=0) == E_SHAPE
    assert _call(lib, n=101, pad=1) == E_SHAPE
    assert _call(lib, n=4096, pad=1) == E_SHAPE
    assert _call(lib, ws_bytes=16) == E_WORKSPACE
    assert _call(lib, ws=257) == E_WORKSPACE
    assert _call(lib, lamb=-1.0) == E_OPTICS
    assert _call(lib, px=float("nan")) == E_OPTICS
    assert _call(lib, in_mode=1) == E_NULL                           # amplitude / phase needs in1


def test_python_rejects_cpu_and_bad_distances():
    import style_transfer_based_holographic_imaging_b200 as pkg
    x = torch.zeros(2, 1, 64, 64, dtype=torch.complex64)
    with pytest.raises(RuntimeError, match="CPU|cpu"):
        pkg.focal_stack(x, [1e-3, 2e-3], LAMB, PX)
    with pytest.raises(RuntimeError, match="CPU|cpu"):
        pkg.autofocus(x.abs(), [1e-3, 2e-3], LAMB, PX)
    from style_transfer_based_holographic_imaging_b200.focus import _stack_distances
    for bad in (torch.zeros(3, 4), torch.zeros(2, 2, 2), torch.zeros(0)):
        with pytest.raises(RuntimeError, match="z must be"):
            _stack_distances(bad, 2, torch.device("cpu"))
    zt, zd, k = _stack_distances(torch.zeros(5, dtype=torch.float32), 2, torch.device("cpu"))
    assert tuple(zt.shape) == (2, 5) and zd == 0 and k == 5
    zt, zd, k = _stack_distances([1e-3, 2e-3], 3, torch.device("cpu"))
    assert tuple(zt.shape) == (3, 2) and zt.dtype == torch.float64 and zd == 1


def test_python_rejects_grad():
    import style_transfer_based_holographic_imaging_b200 as pkg
    x = torch.zeros(1, 64, 64, requires_grad=True)
    with pytest.raises(RuntimeError, match="ASM"):
        pkg.focal_stack(x, [1e-3], LAMB, PX)


def test_focus_metric_formulas():
    from style_transfer_based_holographic_imaging_b200 import focus_metric
    a = torch.rand(3, 50, dtype=torch.float64) + 0.1
    mom = torch.stack([a.sum(1), (a ** 2).sum(1), (a ** 4).sum(1)], dim=1)
    mean, std = a.mean(1), a.std(1, unbiased=False)
    torch.testing.assert_close(focus_metric(mom, 50, "tamura"), torch.sqrt(std / mean))
    i = a ** 2
    torch.testing.assert_close(focus_metric(mom, 50, "variance"), i.var(1, unbiased=False) / i.mean(1) ** 2)
    with pytest.raises(ValueError):
        focus_metric(mom, 50, "tenengrad")
