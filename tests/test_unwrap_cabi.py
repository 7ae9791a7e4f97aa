"""CPU: argument validation of asm_b200_unwrap and its workspace query.  Validation runs before the call touches a device,
so every call here fails on purpose before any launch (an accepted shape is given a workspace one byte short)."""
import ctypes

import pytest

E_NULL, E_SHAPE, E_WORKSPACE = -1, -2, -4
INT_MAX = 2 ** 31 - 1
DUMMY = ctypes.c_void_p(256)          # never dereferenced: validation fails first
HUGE = 1 << 62


@pytest.fixture(scope="module")
def lib():
    from style_transfer_based_holographic_imaging_b200 import build, _lib
    build.build()
    return _lib.load()


def _edges(b, h, w):
    return b * (h * (w - 1) + (h - 1) * w)


SHAPES = [
    (1, 3, 3), (7, 3, 700), (7, 700, 3), (300, 24, 20), (150, 129, 128),          # accepted
    (0, 8, 8), (-1, 8, 8), (1, 2, 8), (1, 8, 2), (1, 0, 0), (1, -3, 3), (4, 2, 2),  # B < 1, H or W < 3
    (1, 1 << 14, 1 << 14), (1, (1 << 14) + 1, 1 << 14), (1, 3, (1 << 28) // 3 + 1),  # H W at and above 2^28
    (1, 1 << 28, 1), (1, INT_MAX, 3), (1, 46341, 46341),                              # H W beyond int
    (1025, 1024, 1024), (1026, 1024, 1024), (600, 1400, 1400), (INT_MAX, 3, 3),     # B E around INT_MAX
]


def _accepted(b, h, w):
    return b >= 1 and h >= 3 and w >= 3 and h * w <= 1 << 28 and _edges(b, h, w) <= INT_MAX


def test_edge_count_limit_lands_where_expected():
    assert _edges(1025, 1024, 1024) <= INT_MAX < _edges(1026, 1024, 1024)
    assert _edges(600, 1400, 1400) > INT_MAX and (1400 * 1400) < 1 << 28


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_workspace_query_is_zero_exactly_for_rejected_shapes(lib, shape):
    b, h, w = shape
    need = lib.asm_b200_unwrap_workspace_bytes(b, h, w)
    if _accepted(b, h, w):
        assert need > 0 and need % 256 == 0
        # the shape passes validation: the next check, the workspace size, is what fails
        assert lib.asm_b200_unwrap(DUMMY, DUMMY, b, h, w, DUMMY, need - 1, None) == E_WORKSPACE
    else:
        assert need == 0
        assert lib.asm_b200_unwrap(DUMMY, DUMMY, b, h, w, DUMMY, HUGE, None) == E_SHAPE


def test_workspace_grows_with_the_batch(lib):
    ws = lib.asm_b200_unwrap_workspace_bytes
    one = ws(1, 129, 128)
    assert ws(150, 129, 128) >= 150 * (129 * 128 * 4 * 5 + _edges(1, 129, 128) * 4 * 6)   # rel/forest + keys/ids/cub
    assert one < ws(2, 129, 128) < ws(150, 129, 128)


def test_null_and_workspace_errors(lib):
    b, h, w = 2, 64, 48
    need = lib.asm_b200_unwrap_workspace_bytes(b, h, w)
    f = lib.asm_b200_unwrap
    assert f(None, DUMMY, b, h, w, DUMMY, need, None) == E_NULL
    assert f(DUMMY, None, b, h, w, DUMMY, need, None) == E_NULL
    assert f(None, DUMMY, 1, 2, 2, DUMMY, need, None) == E_NULL          # pointers are checked before the shape
    assert f(DUMMY, DUMMY, b, h, w, None, need, None) == E_WORKSPACE
    assert f(DUMMY, DUMMY, b, h, w, ctypes.c_void_p(256 + 128), HUGE, None) == E_WORKSPACE   # not 256-byte aligned
    assert f(DUMMY, DUMMY, b, h, w, ctypes.c_void_p(257), HUGE, None) == E_WORKSPACE
    assert f(DUMMY, DUMMY, b, h, w, DUMMY, need - 1, None) == E_WORKSPACE
    assert f(DUMMY, DUMMY, b, h, w, DUMMY, 0, None) == E_WORKSPACE
