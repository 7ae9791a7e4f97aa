"""CPU: the band-limited entry points (asm_b200_*_bl) are exported, reject a band_limit other than 0 or 1 with E_MODE,
and validate every other argument exactly as their counterparts do (the validation cases of test_cabi.py and
test_focus_cabi.py, through the _bl entry points with band_limit 0 and 1).  No compute calls here."""
import ctypes

import pytest

E_NULL, E_SHAPE, E_MODE, E_WORKSPACE, E_OPTICS = -1, -2, -3, -4, -5
LAMB, PX = 532e-9, 1.5e-6
vp = ctypes.c_void_p
D = vp(256)   # never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    from style_transfer_based_holographic_imaging_b200 import build, _lib
    build.build()
    return _lib.load()


def test_exported(lib):
    from style_transfer_based_holographic_imaging_b200 import _lib
    for name in ("forward", "adjoint", "grad_z", "focal_stack"):
        assert hasattr(lib, f"asm_b200_{name}_bl") and f"asm_b200_{name}_bl" in _lib.SYMBOLS
        assert getattr(lib, f"asm_b200_{name}_bl").argtypes == getattr(lib, f"asm_b200_{name}").argtypes + [ctypes.c_int]


# (entry point, arguments of the plain call, expected code): test_cabi.py and test_focus_cabi.py
SINGLE = [
    ("forward", (D, None, D, 0, D, None, 1, 1, 101, 1, 0, 0, LAMB, PX, 1.0, 1.0, D, 1 << 30, None), E_SHAPE),
    ("forward", (D, None, D, 0, D, None, 1, 1, 128, 0, 9, 0, LAMB, PX, 1.0, 1.0, D, 1 << 30, None), E_MODE),
    ("forward", (D, None, D, 0, D, None, 1, 1, 128, 0, 1, 0, LAMB, PX, 1.0, 1.0, D, 1 << 30, None), E_NULL),
    ("forward", (D, None, D, 0, D, None, 1, 1, 128, 0, 0, 0, -1.0, PX, 1.0, 1.0, D, 1 << 30, None), E_OPTICS),
    ("forward", (D, None, D, 0, D, None, 1, 1, 128, 0, 0, 0, LAMB, PX, 1.0, 1.0, D, 16, None), E_WORKSPACE),
    ("forward", (D, None, D, 0, D, None, 1, 1, 128, 0, 0, 0, LAMB, PX, 1.0, 1.0, vp(257), 1 << 30, None), E_WORKSPACE),
    ("forward", (D, None, D, 0, D, None, 1, 2, 128, 0, 0, 3, LAMB, PX, 1.0, 1.0, D, 1 << 30, None), E_MODE),
    ("adjoint", (D, None, D, 0, None, None, D, None, 1, 1, 128, 0, 1, 0, LAMB, PX, 1.0, D, 1 << 30, None), E_MODE),
    ("grad_z", (D, None, D, 0, None, None, 0, D, 1, 1, 128, 0, 0, LAMB, PX, 1.0, D, 1 << 30, None), E_NULL),
]


def _stack(in_mode=0, out_mode=1, out0=256, out1=None, mom=None, k=4, b=1, n=128, pad=0, lamb=LAMB, px=PX, ws=256,
           ws_bytes=1 << 40, in1=None):
    return (D, None if in1 is None else vp(in1), D, 0, k, None if out0 is None else vp(out0),
            None if out1 is None else vp(out1), None if mom is None else vp(mom), b, n, pad, in_mode, out_mode, lamb, px,
            1.0, vp(ws), ws_bytes, None)


STACK = [(dict(out0=None, mom=None), E_NULL), (dict(out_mode=3), E_MODE), (dict(out_mode=5), E_MODE),
         (dict(in_mode=3, in1=256), E_MODE), (dict(in_mode=9), E_MODE), (dict(out_mode=1, out1=256), E_MODE),
         (dict(k=0), E_SHAPE), (dict(b=0), E_SHAPE), (dict(n=101, pad=1), E_SHAPE), (dict(n=4096, pad=1), E_SHAPE),
         (dict(ws_bytes=16), E_WORKSPACE), (dict(ws=257), E_WORKSPACE), (dict(lamb=-1.0), E_OPTICS),
         (dict(px=float("nan")), E_OPTICS), (dict(in_mode=1), E_NULL)]
CASES = SINGLE + [("focal_stack", _stack(**kw), code) for kw, code in STACK]


@pytest.mark.parametrize("i", range(len(CASES)))
def test_validation_matches_counterpart(lib, i):
    name, args, code = CASES[i]
    assert getattr(lib, f"asm_b200_{name}")(*args) == code
    for band_limit in (0, 1):
        assert getattr(lib, f"asm_b200_{name}_bl")(*args, band_limit) == code, (name, band_limit)


@pytest.mark.parametrize("name", ["forward", "adjoint", "grad_z", "focal_stack"])
@pytest.mark.parametrize("band_limit", [2, -1, 1 << 30])
def test_band_limit_out_of_range_is_e_mode(lib, name, band_limit):
    # arguments that the counterpart would accept up to the device check: only band_limit is wrong
    if name == "forward":
        args = (D, None, D, 0, D, None, 1, 1, 128, 0, 0, 0, LAMB, PX, 1.0, 1.0, D, 1 << 30, None)
    elif name == "adjoint":
        args = (D, None, D, 0, None, None, D, None, 1, 1, 128, 0, 0, 0, LAMB, PX, 1.0, D, 1 << 30, None)
    elif name == "grad_z":
        args = (D, None, D, 0, D, None, 0, D, 1, 1, 128, 0, 0, LAMB, PX, 1.0, D, 1 << 30, None)
    else:
        args = _stack()
    assert getattr(lib, f"asm_b200_{name}_bl")(*args, band_limit) == E_MODE
    assert lib.asm_b200_strerror(E_MODE).find(b"band_limit") >= 0
