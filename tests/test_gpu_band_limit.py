"""GPU: the band-limited angular spectrum (asm_b200_*_bl, band_limit=True in Python) on every kernel family.

  - transfer function bin by bin (impulse response, tests/_parity.py): H mask forward, conj(H) mask adjoint, fp32 and
    fp64 distances, B = 2 samples with different limits (about M/4 and 3M/8), C = 2, and a distance whose limit keeps
    every bin;
  - no behaviour change: _bl with band_limit = 0 is the plain entry point bit for bit, and band_limit = 1 at a distance
    whose limit keeps every bin is too;
  - modes against the band-limited float64 oracle at KCAL x the complex64 pipeline's error, grad_z at TOL_GZ;
  - autograd of ASM(..., band_limit=True) and Holo_Generator(args, band_limit=True);
  - focal stacks against single band-limited calls; the launch-sequence graph cache alternating the flag; determinism.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import asm_oracle as ao
import _band_limit as bl
from _parity import (OPTICS, assert_well_conditioned, check_field, check_grad_z, check_transfer, empty_device, polar,
                     recover_h, to_device)

pytestmark = pytest.mark.gpu

LAMB, PX = OPTICS["default"]


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as p
    p._lib.load()
    return p


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _zd(L, z):
    return L.Z_F64 if z.dtype == torch.float64 else L.Z_F32


def _ws(lib, b, c, n, pad):
    return torch.empty(lib.asm_b200_workspace_bytes(b, c, n, int(pad)), dtype=torch.uint8, device="cuda")


def fwd(L, in0, in1, z, out0, out1, b, c, n, pad, in_mode, out_mode, band_limit, in_scale=1.0, out_scale=1.0):
    """asm_b200_forward_bl(..., band_limit), or the plain asm_b200_forward for band_limit=None."""
    lib = L.load()
    ws = _ws(lib, b, c, n, pad)
    args = (_p(in0), _p(in1), _p(z), _zd(L, z), _p(out0), _p(out1), b, c, n, int(pad), in_mode, out_mode, LAMB, PX,
            in_scale, out_scale, _p(ws), ws.numel(), _st())
    L.check(lib.asm_b200_forward(*args) if band_limit is None else lib.asm_b200_forward_bl(*args, band_limit))


def adj(L, in0, in1, z, aux0, aux1, out0, out1, b, c, n, pad, in_mode, out_mode, band_limit, in_scale=1.0):
    lib = L.load()
    ws = _ws(lib, b, c, n, pad)
    args = (_p(in0), _p(in1), _p(z), _zd(L, z), _p(aux0), _p(aux1), _p(out0), _p(out1), b, c, n, int(pad), in_mode,
            out_mode, LAMB, PX, in_scale, _p(ws), ws.numel(), _st())
    L.check(lib.asm_b200_adjoint(*args) if band_limit is None else lib.asm_b200_adjoint_bl(*args, band_limit))


def gradz(L, in0, in1, z, cot0, cot1, cot_mode, out, b, c, n, pad, in_mode, band_limit, in_scale=1.0):
    lib = L.load()
    ws = _ws(lib, b, c, n, pad)
    args = (_p(in0), _p(in1), _p(z), _zd(L, z), _p(cot0), _p(cot1), cot_mode, _p(out), b, c, n, int(pad), in_mode,
            LAMB, PX, in_scale, _p(ws), ws.numel(), _st())
    L.check(lib.asm_b200_grad_z(*args) if band_limit is None else lib.asm_b200_grad_z_bl(*args, band_limit))


def _np(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _zpair(m, dtype):
    """Two distances whose limits differ: about M/4 and 3M/8 (both well inside M/2)."""
    return np.array([bl.z_for_lim(m, LAMB, PX, m // 4), bl.z_for_lim(m, LAMB, PX, 3 * m // 8)]).astype(dtype)


def _zfull(m, dtype):
    """A distance whose limit keeps every bin (lim >= M/2)."""
    z = np.array([bl.z_for_lim(m, LAMB, PX, m // 2 + 2)]).astype(dtype)
    assert bl.band_limit_mask(m, LAMB, PX, z)[0][0] >= m // 2
    return z


# --------------------------------------------------------------------------------------------
# transfer function, bin by bin
# --------------------------------------------------------------------------------------------
SIZES = [32, 64, 128, 256, 512, 1024, 2048, 4096, 45, 92, 250, 1000]
# (operation, input offset, output offset, z dtype): bulk (aligned) and register (offset) row kernels on both sides
VARIANTS = [("fwd", 0, 0, np.float32), ("fwd", 1, 1, np.float64), ("adj", 0, 0, np.float64), ("adj", 1, 1, np.float32)]


def _impulse_h(pkg, op, off_in, off_out, z, n, band_limit, c=2):
    L = pkg._lib
    b = len(z)
    imp = np.zeros((b, c, n, n), dtype=np.complex64)
    imp[:, :, 0, 0] = 1.0
    x = to_device(imp, off_in)
    zt = torch.from_numpy(z).cuda()
    out = empty_device((b, c, n, n), torch.complex64, off_out)
    if op == "fwd":
        fwd(L, x, None, zt, out, None, b, c, n, 0, ao.IN_COMPLEX, ao.OUT_COMPLEX, band_limit)
    else:
        adj(L, x, None, zt, None, None, out, None, b, c, n, 0, ao.IN_COMPLEX, ao.OUT_COMPLEX, band_limit)
    return _np(out)


@pytest.mark.parametrize("n", SIZES)
def test_transfer_function_per_bin(pkg, n):
    m = n
    zmax = float(np.abs(_zpair(m, np.float64)).max())
    assert_well_conditioned(m, m, LAMB, PX, zmax)
    for op, off_in, off_out, dt in VARIANTS:
        z = _zpair(m, dt)
        lims = bl.band_limit_mask(m, LAMB, PX, z)[0]
        assert lims[0] != lims[1] and lims.max() < m // 2
        ref = bl.h_bl(m, m, LAMB, PX, z)
        ref = np.conj(ref) if op == "adj" else ref
        h = recover_h(_impulse_h(pkg, op, off_in, off_out, z, n, 1))
        for c in range(h.shape[1]):
            check_transfer(h[:, c], ref, f"{op} off({off_in},{off_out}) {np.dtype(dt).name} lims {lims.tolist()} ch {c}")
    # a limit that keeps every bin: the plain H on all bins
    z = _zfull(m, np.float32)
    ref = ao.transfer_function(m, m, LAMB, PX, z)
    check_transfer(recover_h(_impulse_h(pkg, "fwd", 0, 0, z, n, 1, c=1))[:, 0], ref, "fwd full band")


# --------------------------------------------------------------------------------------------
# no behaviour change
# --------------------------------------------------------------------------------------------
# (N, pad, buffer offset): generic <= 512, k32t 1024, k64 2048 with the warp-pair (aligned) and generic (offset) row
# kernels, on-the-fly H at 4096, and the matrix-product path
FAMILIES = [(64, False, 0), (256, False, 0), (1024, False, 0), (512, True, 0), (2048, False, 0), (2048, False, 1),
            (4096, False, 0), (45, False, 0), (92, True, 0)]


@pytest.mark.parametrize("n,pad,off", FAMILIES, ids=[f"{n}{'p' if p else ''}-off{o}" for n, p, o in FAMILIES])
def test_no_behaviour_change(pkg, n, pad, off):
    L = pkg._lib
    m = bl.fft_size(n, pad)
    b, c = (1, 2) if m >= 2048 else (2, 2)
    rng = np.random.default_rng(n + off)
    shape = (b, c, n, n)
    o = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    g = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    x, gt = to_device(o, off), to_device(g, off)
    z_bite = torch.from_numpy(_zpair(m, np.float32)[:b]).cuda()
    z_full = torch.from_numpy(np.repeat(_zfull(m, np.float64), b)).cuda()

    def run(kind, z, flag):
        if kind == "grad":
            out = torch.empty(b, dtype=torch.float64, device="cuda")
            gradz(L, x, None, z, gt, None, ao.IN_COMPLEX, out, b, c, n, pad, ao.IN_COMPLEX, flag)
            return _np(out)
        out = empty_device(shape, torch.complex64, off)
        if kind == "fwd":
            fwd(L, x, None, z, out, None, b, c, n, pad, ao.IN_COMPLEX, ao.OUT_COMPLEX, flag)
        else:
            adj(L, gt, None, z, None, None, out, None, b, c, n, pad, ao.IN_COMPLEX, ao.OUT_COMPLEX, flag)
        return _np(out)

    for kind in ("fwd", "adj"):
        plain = run(kind, z_bite, None)
        assert np.array_equal(run(kind, z_bite, 0), plain), kind
        assert not np.array_equal(run(kind, z_bite, 1), plain), kind          # the limit bites at these distances
        assert np.array_equal(run(kind, z_full, 1), run(kind, z_full, None)), kind
    # grad_z sums with double atomics (order not fixed): equal to rounding
    for z in (z_bite, z_full):
        a, bb = run("grad", z, None), run("grad", z, 0)
        assert np.allclose(a, bb, rtol=1e-9, atol=0), (a, bb)
    a, bb = run("grad", z_full, None), run("grad", z_full, 1)
    assert np.allclose(a, bb, rtol=1e-9, atol=0), (a, bb)
    # focal stack
    if not off:
        zs = torch.from_numpy(np.stack([_zpair(m, np.float32)] * b)).cuda()
        lib = L.load()
        k = zs.shape[1]
        need = lib.asm_b200_focal_stack_workspace_bytes(b, k, n, int(pad))
        ws = torch.empty(need, dtype=torch.uint8, device="cuda")
        xs = x[:, 0].contiguous()
        outs = []
        for flag in (None, 0):
            out = torch.empty((b, k, n, n), dtype=torch.complex64, device="cuda")
            mom = torch.empty((b, k, 3), dtype=torch.float64, device="cuda")
            args = (_p(xs), None, _p(zs), L.Z_F32, k, _p(out), None, _p(mom), b, n, int(pad), ao.IN_COMPLEX,
                    ao.OUT_COMPLEX, LAMB, PX, 1.0, _p(ws), need, _st())
            L.check(lib.asm_b200_focal_stack(*args) if flag is None else lib.asm_b200_focal_stack_bl(*args, flag))
            outs.append((_np(out), _np(mom)))
        assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])


# --------------------------------------------------------------------------------------------
# modes against the oracle
# --------------------------------------------------------------------------------------------
MODE_SIZES = [(64, False), (32, True), (256, False), (1024, False), (512, True), (2048, False), (4096, False), (92, True)]
OUT_MODES = [(ao.OUT_COMPLEX, False), (ao.OUT_INTENSITY, False), (ao.OUT_INTENSITY, True), (ao.OUT_ABS_ANGLE, True),
             (ao.OUT_ABSANG_CAT, False)]
IN_SCALE, OUT_SCALE = 0.7, 1.7


@pytest.mark.parametrize("n,pad", MODE_SIZES, ids=[f"{n}{'p' if p else ''}" for n, p in MODE_SIZES])
def test_modes_against_oracle(pkg, n, pad):
    L = pkg._lib
    m = bl.fft_size(n, pad)
    b, c = (1, 2) if m >= 2048 else (2, 2)
    rng = np.random.default_rng(7 * n + pad)
    shape = (b, c, n, n)
    for zdt in (np.float32, np.float64):
        z = _zpair(m, zdt)[:b] if b == 2 else _zpair(m, zdt)[1:]
        zt = torch.from_numpy(z).cuda()
        o = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
        x = to_device(o)
        ref = bl.propagate(o, LAMB, z, PX, pad)
        c64 = bl.propagate(o, LAMB, z, PX, pad, dtype=np.complex64)
        what = f"N={n} pad={pad} {np.dtype(zdt).name}"
        for out_mode, with_out1 in OUT_MODES:
            tag = f"{what} fwd out{out_mode}{'+U' if with_out1 else ''}"
            if out_mode == ao.OUT_ABSANG_CAT:                                     # C must be 1
                zc = torch.repeat_interleave(zt, c)
                out0 = empty_device((b * c, 2, n, n), torch.float32)
                fwd(L, x, None, zc, out0, None, b * c, 1, n, pad, ao.IN_COMPLEX, out_mode, 1, 1.0, OUT_SCALE)
                k = _np(out0)
                e = ao.output_stage(c64.reshape(b * c, 1, n, n), out_mode, OUT_SCALE)[0]
                check_field(polar(k[:, 0], k[:, 1]), ref.reshape(b * c, n, n) * OUT_SCALE, polar(e[:, 0], e[:, 1]), tag)
                continue
            out0 = empty_device(shape, torch.complex64 if out_mode == ao.OUT_COMPLEX else torch.float32)
            out1 = None
            if with_out1:
                out1 = empty_device(shape, torch.complex64 if out_mode == ao.OUT_INTENSITY else torch.float32)
            fwd(L, x, None, zt, out0, out1, b, c, n, pad, ao.IN_COMPLEX, out_mode, 1)
            e = ao.output_stage(c64, out_mode)
            if out_mode == ao.OUT_COMPLEX:
                check_field(_np(out0), ref, e[0], tag)
            elif out_mode == ao.OUT_INTENSITY:
                check_field(_np(out0), np.abs(ref) ** 2, e[0], tag)
                if with_out1:
                    check_field(_np(out1), ref, e[1], tag + " out1")
            else:
                check_field(polar(_np(out0), _np(out1)), ref, polar(e[0], e[1]), tag)
        # adjoint: COMPLEX and GRAD_AP
        g = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
        gt = to_device(g)
        aref = bl.propagate(g, LAMB, z, PX, pad, adjoint=True)
        a64 = bl.propagate(g, LAMB, z, PX, pad, adjoint=True, dtype=np.complex64)
        out0 = empty_device(shape, torch.complex64)
        adj(L, gt, None, zt, None, None, out0, None, b, c, n, pad, ao.IN_COMPLEX, ao.OUT_COMPLEX, 1)
        check_field(_np(out0), aref, a64, f"{what} adj COMPLEX")
        amp = rng.uniform(0.2, 1.5, shape).astype(np.float32)
        ph = rng.uniform(-np.pi, np.pi, shape).astype(np.float32)
        ga, gp = empty_device(shape, torch.float32), empty_device(shape, torch.float32)
        adj(L, gt, None, zt, to_device(amp), to_device(ph), ga, gp, b, c, n, pad, ao.IN_COMPLEX, ao.OUT_GRAD_AP, 1,
            IN_SCALE)
        r, e = ao.grad_ap(aref, amp, ph, IN_SCALE), ao.grad_ap(a64, amp, ph, IN_SCALE)
        check_field(_np(ga), r[0], e[0], f"{what} adj GRAD_AP dA")
        check_field(_np(gp), r[1], e[1], f"{what} adj GRAD_AP dphase")
        # grad_z, both cotangents
        u, du = bl.dudz(o, LAMB, z, PX, pad)
        for cot_mode in (ao.IN_COMPLEX, ao.IN_COT_FIELD):
            if cot_mode == ao.IN_COMPLEX:
                gg, kshift, cot = g.astype(np.complex128), 0.0, (gt, None)
            else:
                w = rng.uniform(-1.0, 1.0, shape).astype(np.float32)
                uu = u.astype(np.complex64)
                gg, kshift, cot = 2.0 * w.astype(np.float64) * uu, 1.0, (to_device(w), to_device(uu))
            want, scale = ao.grad_z_sum(gg, u, du, LAMB, z, kshift)
            got = torch.empty(b, dtype=torch.float64, device="cuda")
            gradz(L, x, None, zt, cot[0], cot[1], cot_mode, got, b, c, n, pad, ao.IN_COMPLEX, 1)
            check_grad_z(_np(got), want, scale, f"{what} cot{cot_mode}")


# --------------------------------------------------------------------------------------------
# autograd
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,pad", [(256, False), (64, True)])
def test_asm_autograd(pkg, n, pad):
    m = bl.fft_size(n, pad)
    rng = np.random.default_rng(21)
    shape = (2, 1, n, n)
    o = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    g = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
    z = _zpair(m, np.float32).reshape(2, 1, 1, 1)
    O = torch.from_numpy(o).cuda().requires_grad_(True)
    d = torch.from_numpy(z).cuda().requires_grad_(True)
    U = pkg.ASM(O, LAMB, d, PX, zero_padding=pad, band_limit=True)
    gO, gd = torch.autograd.grad(torch.real(torch.sum(torch.conj(torch.from_numpy(g).cuda()) * U)), [O, d])
    ref = bl.propagate(o, LAMB, z.reshape(-1), PX, pad)
    assert ao.rel_l2(_np(U.detach()), ref) < 1e-5
    assert ao.rel_l2(_np(gO), bl.propagate(g, LAMB, z.reshape(-1), PX, pad, adjoint=True)) < 1e-5
    u, du = bl.dudz(o, LAMB, z.reshape(-1), PX, pad)
    want, scale = ao.grad_z_sum(g, u, du, LAMB, z.reshape(-1))
    assert gd.shape == d.shape
    check_grad_z(_np(gd).reshape(-1), want, scale, "ASM band_limit")
    # the plain call differs at these distances
    assert ao.rel_l2(_np(pkg.ASM(O.detach(), LAMB, d.detach(), PX, zero_padding=pad)), ref) > 1e-2


def test_holo_generator_autograd(pkg):
    n = 128
    args = ao.Optics(phase_normalize=1.3)
    rng = np.random.default_rng(22)
    shape = (2, 1, n, n)
    amp = rng.uniform(0.3, 1.0, shape).astype(np.float32)
    ph = rng.uniform(-np.pi, np.pi, shape).astype(np.float32)
    w = rng.standard_normal(shape).astype(np.float32)
    dmm = (_zpair(2 * n, np.float64) * 1e3).astype(np.float32).reshape(2, 1, 1, 1)   # mm, as the reference's d
    z = ao.metres(dmm, args).reshape(-1)
    assert np.all(bl.band_limit_mask(2 * n, LAMB, PX, z)[0] < n)
    hg = pkg.Holo_Generator(args, band_limit=True)
    A = torch.from_numpy(amp).cuda().requires_grad_(True)
    P = torch.from_numpy(ph).cuda().requires_grad_(True)
    D = torch.from_numpy(dmm).cuda().requires_grad_(True)
    I = hg(A, P, D)
    gA, gP, gD = torch.autograd.grad(torch.sum(torch.from_numpy(w).cuda() * I), [A, P, D])
    o = ao.object_field(amp, ph, args)
    u, du = bl.dudz(o, LAMB, z, PX, True)
    g = 2.0 * w.astype(np.float64) * u
    go = bl.propagate(g, LAMB, z, PX, True, adjoint=True)
    e = np.exp(1j * (ph * np.float32(args.phase_normalize)).astype(np.float64))
    want_d, scale = ao.grad_z_sum(g, u, du, LAMB, z)
    k = float(np.float32(args.distance_normalize)) * float(np.float32(1e-3))
    assert ao.rel_l2(_np(I.detach()), np.abs(u) ** 2) < 1e-5
    assert ao.rel_l2(_np(gA), np.real(np.conj(e) * go)) < 1e-4
    assert ao.rel_l2(_np(gP), args.phase_normalize * np.imag(np.conj(o) * go)) < 1e-4
    check_grad_z(_np(gD).reshape(-1) / k, want_d, scale, "Holo_Generator band_limit")


# --------------------------------------------------------------------------------------------
# focal stacks, graph cache, determinism
# --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,pad", [(1024, False), (2048, False), (92, True)])
def test_focal_stack_matches_single_calls(pkg, n, pad):
    m = bl.fft_size(n, pad)
    rng = np.random.default_rng(23)
    b = 2
    x = torch.from_numpy((rng.standard_normal((b, n, n)) + 1j * rng.standard_normal((b, n, n))).astype(np.complex64)).cuda()
    zk = np.concatenate([_zpair(m, np.float32), _zfull(m, np.float32)])
    z = torch.from_numpy(np.stack([zk, zk[::-1].copy()])).cuda()                    # [B, K], each plane its own limit
    img, mom = pkg.focal_stack(x, z, LAMB, PX, pad, output="complex", moments=True, band_limit=True)
    for k in range(z.shape[1]):
        one = pkg.asm_forward_raw(x[:, None], z[:, k].reshape(b, 1, 1, 1), LAMB, PX, pad, band_limit=True)[:, 0]
        r = ao.rel_l2(_np(img[:, k]), _np(one))
        assert r <= 2e-6, (k, r)
        a = one.abs().to(torch.float64).reshape(b, -1)
        mref = torch.stack([a.sum(-1), (a ** 2).sum(-1), (a ** 4).sum(-1)], -1)
        assert float(((mom[:, k] - mref).abs() / mref).max()) < 1e-5
    plain = pkg.focal_stack(x, z, LAMB, PX, pad, output="complex")
    assert ao.rel_l2(_np(plain[:, 0]), _np(img[:, 0])) > 1e-2                     # the limit bites on plane 0


def test_graph_cache_keys_on_the_flag(pkg):
    """FFT 256, 256 samples: enough chunks for the launch-sequence cache; identical pointers, the flag alternating."""
    L = pkg._lib
    lib = L.load()
    n, b = 256, 256
    rng = np.random.default_rng(24)
    o = (rng.standard_normal((b, 1, n, n)) + 1j * rng.standard_normal((b, 1, n, n))).astype(np.complex64)
    x = torch.from_numpy(o).cuda()
    z = np.full(b, bl.z_for_lim(n, LAMB, PX, n // 4), dtype=np.float32)
    zt = torch.from_numpy(z).cuda()
    out = torch.empty((b, 1, n, n), dtype=torch.complex64, device="cuda")
    ws = _ws(lib, b, 1, n, False)
    pick = [0, 1, b - 1]
    refs = {flag: bl.propagate(o[pick], LAMB, z[pick], PX, band_limit=bool(flag)) for flag in (0, 1)}
    c64s = {flag: bl.propagate(o[pick], LAMB, z[pick], PX, band_limit=bool(flag), dtype=np.complex64) for flag in (0, 1)}
    first = {}
    for i, flag in enumerate([0, 1, 0, 1, 0, 1, 0, 1]):
        L.check(lib.asm_b200_forward_bl(_p(x), None, _p(zt), L.Z_F32, _p(out), None, b, 1, n, 0, ao.IN_COMPLEX,
                                        ao.OUT_COMPLEX, LAMB, PX, 1.0, 1.0, _p(ws), ws.numel(), _st(), flag))
        res = _np(out)
        check_field(res[pick], refs[flag], c64s[flag], f"call {i} band_limit={flag}")
        if flag in first:
            assert np.array_equal(res, first[flag]), i
        else:
            first[flag] = res


@pytest.mark.parametrize("n,pad", [(1024, False), (2048, False), (512, True), (92, True)])
def test_repeated_calls_bit_identical(pkg, n, pad):
    m = bl.fft_size(n, pad)
    rng = np.random.default_rng(25)
    x = torch.from_numpy((rng.standard_normal((2, 1, n, n)) + 1j * rng.standard_normal((2, 1, n, n))).astype(np.complex64)).cuda()
    z = torch.from_numpy(_zpair(m, np.float32).reshape(2, 1, 1, 1)).cuda()
    runs = [pkg.asm_forward_raw(x, z, LAMB, PX, pad, band_limit=True) for _ in range(3)]
    runs += [pkg.asm_adjoint_raw(x, z, LAMB, PX, pad, band_limit=True) for _ in range(2)]
    torch.cuda.synchronize()
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2]) and torch.equal(runs[3], runs[4])
