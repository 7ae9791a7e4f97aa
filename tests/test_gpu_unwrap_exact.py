"""Device phase unwrapping (asm_b200_unwrap) pinned to the CPU oracle (oracle/unwrap_oracle.py) pixel for pixel.

The oracle computes the same fp32 reliabilities and keys, sorts stably with the same tie order and merges with the same
rules, so on every pixel the kernel's 2 pi increment must equal the oracle's and its value must equal
``unwrap_oracle.compose`` bit for bit.  The cases (tests/_unwrap_cases.py) are the ones tests/test_unwrap_power.py shows can
tell planted defects apart.  Shapes cover both merge kernels: up to 128 x 128 = 16384 pixels the forest lives in shared
memory (k_unwrap_merge_smem), above that in global memory (k_unwrap_merge)."""
import functools

import numpy as np
import pytest
import torch

import _unwrap_cases as uc
from oracle import asm_oracle as ao
from oracle import unwrap_oracle as uo

pytestmark = pytest.mark.gpu

SMEM_PIX = 16384
SMEM_SHAPES = [(3, 3), (3, 700), (700, 3), (64, 48), (127, 129), (128, 128)]
GLOBAL_SHAPES = [(129, 128), (5, 3277), (3, 6000), (200, 333), (256, 256)]


def _id(shape):
    h, w = shape
    return f"{h}x{w}-{'smem' if h * w <= SMEM_PIX else 'global'}"


@pytest.fixture(scope="module")
def pkg():
    import style_transfer_based_holographic_imaging_b200 as p
    return p


@functools.lru_cache(maxsize=None)
def _case_inc(name, h, w):
    return uo.increments(uc.case(name, h, w))


def _batch_inc(h, w):
    return np.stack([_case_inc(n, h, w) for n in uc.NAMES])


def _assert_exact(got, ph, inc, label):
    """got, ph: fp32 [..., H, W]; inc: the oracle's increments of ph."""
    got = np.asarray(got, dtype=np.float32).reshape(inc.shape)
    ph = np.asarray(ph, dtype=np.float32).reshape(inc.shape)
    k = np.round((got.astype(np.float64) - ph.astype(np.float64)) / (2 * np.pi)).astype(np.int64)
    bad = k != inc
    assert not bad.any(), f"{label}: {int(bad.sum())} of {bad.size} increments differ, first at {np.argwhere(bad)[0]}"
    want = uo.compose(ph, inc)
    diff = got.view(np.int32) != want.view(np.int32)
    assert not diff.any(), f"{label}: {int(diff.sum())} values differ in their bits, first at {np.argwhere(diff)[0]}"


def _unwrap(pkg, x):
    out = pkg.unwrap(x)
    assert out.dtype == torch.float32 and out.is_cuda
    return out.cpu().numpy()


@pytest.mark.parametrize("shape", SMEM_SHAPES + GLOBAL_SHAPES, ids=_id)
def test_every_case_matches_oracle(pkg, shape):
    h, w = shape
    x = uc.batch(h, w)
    got = _unwrap(pkg, torch.from_numpy(x[:, None]).cuda())
    assert got.shape == (len(uc.NAMES), 1, h, w)
    for i, name in enumerate(uc.NAMES):
        _assert_exact(got[i], x[i], _case_inc(name, h, w), f"{name} {h}x{w}")


@pytest.mark.parametrize("shape", [(64, 48), (129, 128)], ids=_id)
def test_single_image(pkg, shape):
    """B = 1, given as [H, W]."""
    h, w = shape
    for name in uc.NAMES:
        x = uc.case(name, h, w)
        got = _unwrap(pkg, torch.from_numpy(x).cuda())
        assert got.shape == (1, 1, h, w)
        _assert_exact(got, x, _case_inc(name, h, w), f"{name} {h}x{w}")


@pytest.mark.parametrize("b,h,w", [(300, 24, 20), (150, 129, 128)], ids=["300x24x20-smem", "150x129x128-global"])
def test_large_batch(pkg, b, h, w):
    """Image i is case i mod 7, so neighbouring images always differ and a mix-up between samples shows.  At 24 x 20 the
    shared-memory merge runs one block per SM: 300 images are three waves on 148 SMs."""
    pick = np.arange(b) % len(uc.NAMES)
    x = uc.batch(h, w)[pick]
    got = _unwrap(pkg, torch.from_numpy(x).cuda())
    _assert_exact(got, x, _batch_inc(h, w)[pick], f"B={b} {h}x{w}")


def test_tiny_searched_cases(pkg):
    for name, (seed, kind) in uc.TINY.items():
        x = uc.tiny(seed, kind)
        _assert_exact(_unwrap(pkg, torch.from_numpy(x).cuda()), x, uo.increments(x), name)


def test_input_layouts_and_dtypes(pkg):
    h, w = 40, 36
    x = uc.batch(h, w)
    inc = np.stack([uo.increments(im) for im in x])
    t = torch.from_numpy(x).cuda()
    _assert_exact(_unwrap(pkg, t), x, inc, "[B, H, W]")
    _assert_exact(_unwrap(pkg, t[:, None]), x, inc, "[B, 1, H, W]")
    tt = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).cuda().transpose(1, 2)
    assert not tt.is_contiguous() and torch.equal(tt, t)
    _assert_exact(_unwrap(pkg, tt), x, inc, "transposed view")
    _assert_exact(_unwrap(pkg, t.clone().requires_grad_(True)), x, inc, "requires_grad")
    x64 = x.astype(np.float64) + np.random.default_rng(1).uniform(-1e-7, 1e-7, x.shape)   # not representable in fp32
    x32 = x64.astype(np.float32)
    _assert_exact(_unwrap(pkg, torch.from_numpy(x64).cuda()), x32, np.stack([uo.increments(im) for im in x32]), "fp64")


def _abi_unwrap(pkg, ph, out, b, h, w, ws):
    lib = pkg._lib.load()
    rc = lib.asm_b200_unwrap(ph.data_ptr(), out.data_ptr(), b, h, w, ws.data_ptr(), ws.numel(),
                             torch.cuda.current_stream().cuda_stream)
    pkg._lib.check(rc)


@pytest.mark.parametrize("shape", [(64, 48), (129, 128)], ids=_id)
def test_in_place(pkg, shape):
    """out == phase, which include/asm_b200.h allows."""
    h, w = shape
    x = uc.batch(h, w)
    t = torch.from_numpy(x).cuda()
    ws = torch.empty(pkg._lib.load().asm_b200_unwrap_workspace_bytes(len(x), h, w), dtype=torch.uint8, device="cuda")
    _abi_unwrap(pkg, t, t, len(x), h, w, ws)
    _assert_exact(t.cpu().numpy(), x, _batch_inc(h, w), f"in place {h}x{w}")


@pytest.mark.parametrize("sx,sy", [((64, 48), (129, 128)), ((129, 128), (127, 129))], ids=["smem-then-global",
                                                                                           "global-then-smem"])
def test_workspace_reuse(pkg, sx, sy):
    """X, then Y, then X again in one workspace, each into an output filled with NaN: the second X must equal the first
    bit for bit (nothing left by an earlier call is read)."""
    lib = pkg._lib.load()
    x, y = uc.batch(*sx), uc.batch(*sy)
    need = max(lib.asm_b200_unwrap_workspace_bytes(len(x), *sx), lib.asm_b200_unwrap_workspace_bytes(len(y), *sy))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    tx, ty = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
    outs = []
    for t, (h, w) in [(tx, sx), (ty, sy), (tx, sx)]:
        out = torch.full_like(t, float("nan"))
        _abi_unwrap(pkg, t, out, len(t), h, w, ws)
        outs.append(out.cpu().numpy())
    _assert_exact(outs[0], x, _batch_inc(*sx), "X first")
    _assert_exact(outs[1], y, _batch_inc(*sy), "Y")
    assert np.array_equal(outs[0].view(np.int32), outs[2].view(np.int32))


def test_side_stream(pkg):
    """The phase comes from holo_abs_angle on a side stream and is unwrapped there with no sync in between."""
    from style_transfer_based_holographic_imaging_b200 import functional as F_
    rng = np.random.default_rng(8)
    b, n = 6, 128
    args = ao.Optics()
    amp = torch.full((b, 1, n, n), 0.6, device="cuda")
    ph = torch.from_numpy((rng.random((b, 1, n, n)) * 4.0).astype(np.float32)).cuda()
    z = torch.from_numpy(rng.uniform(-3e-4, -1e-4, (b, 1, 1, 1)).astype(np.float32)).cuda()
    call = lambda: F_.holo_abs_angle(amp, ph, z, args.wavelength, args.pixel_size, args.phase_normalize, True)[1]
    ang0 = call()
    un0 = F_.unwrap_phase(ang0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        un1 = F_.unwrap_phase(call())
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(un0, un1)
    a = ang0.cpu().numpy()
    _assert_exact(un0.cpu().numpy(), a, np.stack([uo.increments(im) for im in a[:, 0]]), "holo_abs_angle phase")


@pytest.mark.parametrize("n", [128, 92])
def test_back_focus_unwrap(pkg, n):
    """Holo_Generator(..., return_field=True, unwrap=True) against the oracle run on the same call's unwrap=False angle."""
    rng = np.random.default_rng(9)
    b = 3
    amp = np.full((b, 1, n, n), 0.6, dtype=np.float32)
    ph = np.zeros((b, 1, n, n), dtype=np.float32)
    lo, hi = n * 5 // 16, n * 11 // 16
    ph[:, :, lo:hi, lo:hi] = rng.random((b, 1, hi - lo, hi - lo)).astype(np.float32)
    d = np.full((b, 1, 1, 1), -0.2, dtype=np.float32)
    hg = pkg.Holo_Generator(ao.Optics()).cuda()
    A, P, D = (torch.from_numpy(v).cuda() for v in (amp, ph, d))
    with torch.no_grad():
        a0, p0 = hg(A, P, D, return_field=True)
        a1, p1 = hg(A, P, D, return_field=True, unwrap=True)
    assert torch.equal(a0, a1) and p1.shape == p0.shape
    ang = p0.cpu().numpy()
    _assert_exact(p1.cpu().numpy(), ang, np.stack([uo.increments(im) for im in ang[:, 0]]), f"back focus N={n}")


def test_unsupported_shape_is_refused_before_allocating(pkg):
    """600 images of 1400 x 1400 have more edges than an int counts: refused before the 80 GB workspace is allocated."""
    x = torch.zeros((1, 1, 1400, 1400), device="cuda").expand(600, 1, 1400, 1400)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    before = torch.cuda.memory_allocated()
    with pytest.raises(RuntimeError, match="unsupported shape"):
        pkg.unwrap(x)
    assert torch.cuda.max_memory_allocated() - before < 1 << 20
