"""GPU: every combination the C ABI accepts, on every kernel family, against the float64 oracle.

  forward : the 6 in_modes x {COMPLEX, INTENSITY with and without out1, ABS_ANGLE, REIM_CAT, ABSANG_CAT}
  adjoint : {COMPLEX, COT_FIELD} x {COMPLEX, GRAD_AP}
  grad_z  : the 6 in_modes x the 2 cotangent modes
on one unpadded and one padded size per family (64 / 32p, 256 / 128p, 1024 / 512p, 2048 / 1024p, 4096 / 2048p, and the
matrix-product path at 45 and 92p), with C > 1 wherever the mode allows it, both distance dtypes, default and ring
optics, buffers offset by one element at FFT 1024 and 2048 (the register row kernels), and input phases on both sides
of the +-5e4 switch of the sin / cos reduction.

Bounds (tests/_parity.py): a field output may be at most KCAL times further from the float64 oracle than a plain
complex64 pipeline is (angles are compared through |U| e^{i angle}); a distance gradient at most TOL_GZ * S_b away,
S_b = sum |Re(conj(g) dU/dz)| being the rounding scale of the sum.  Every case prints its error next to its bound.
"""
import numpy as np
import pytest
import torch

from oracle import asm_oracle as ao
from _parity import (KCAL, OPTICS, abi_adjoint, abi_forward, abi_grad_z, check_field, check_grad_z, empty_device, polar,
                     random_inputs, to_device)

pytestmark = pytest.mark.gpu

IN_SCALE = 0.7
OUT_SCALE = 1.7
IN_MODES = [ao.IN_COMPLEX, ao.IN_AMP_PHASE, ao.IN_SQRT_REAL, ao.IN_COT_FIELD, ao.IN_REAL, ao.IN_CONST_AMP_PHASE]
# (out_mode, with out1)
OUT_MODES = [(ao.OUT_COMPLEX, False), (ao.OUT_INTENSITY, False), (ao.OUT_INTENSITY, True), (ao.OUT_ABS_ANGLE, True),
             (ao.OUT_REIM_CAT, False), (ao.OUT_ABSANG_CAT, False)]

SIZES = [(64, False), (32, True), (256, False), (128, True), (1024, False), (512, True), (2048, False), (1024, True),
         (4096, False), (2048, True), (45, False), (92, True)]
# FFT 4096 (the most expensive oracle) with one optics per size; every other size with both
CASES = [(n, pad, o) for n, pad in SIZES for o in ("default", "ring") if not ((2 * n if pad else n) == 4096 and
                                                                          (o == "ring") != pad)]


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as p
    p._lib.load()
    return p


def _np(t):
    return t.cpu().numpy()


def _check_forward(L, inp, zt, ref, c64, b, c, n, pad, in_mode, lamb, px, off):
    in0, in1 = inp
    ratios = []
    for out_mode, with_out1 in OUT_MODES:
        what = f"fwd in{in_mode} out{out_mode}{'+U' if with_out1 else ''}"
        if out_mode in (ao.OUT_REIM_CAT, ao.OUT_ABSANG_CAT):     # C must be 1: the same planes as B*C samples
            bb, cc, zc = b * c, 1, torch.repeat_interleave(zt, c)
            out0 = empty_device((bb, 2, n, n), torch.float32, off)
            abi_forward(L, in0, in1, zc, out0, None, bb, cc, n, pad, in_mode, out_mode, lamb, px, IN_SCALE, OUT_SCALE)
            torch.cuda.synchronize()
            k = _np(out0)
            r = ref.reshape(bb, 1, n, n) * OUT_SCALE
            e = ao.output_stage(c64.reshape(bb, 1, n, n), out_mode, OUT_SCALE)[0]
            if out_mode == ao.OUT_REIM_CAT:
                ratios.append(check_field(k[:, 0] + 1j * k[:, 1], r[:, 0], e[:, 0] + 1j * e[:, 1], what))
            else:
                ratios.append(check_field(polar(k[:, 0], k[:, 1]), r[:, 0], polar(e[:, 0], e[:, 1]), what))
            continue
        out0 = empty_device((b, c, n, n), torch.complex64 if out_mode == ao.OUT_COMPLEX else torch.float32, off)
        out1 = None
        if with_out1:
            out1 = empty_device((b, c, n, n), torch.complex64 if out_mode == ao.OUT_INTENSITY else torch.float32, off)
        abi_forward(L, in0, in1, zt, out0, out1, b, c, n, pad, in_mode, out_mode, lamb, px, IN_SCALE, OUT_SCALE)
        torch.cuda.synchronize()
        e = ao.output_stage(c64, out_mode)
        if out_mode == ao.OUT_COMPLEX:
            ratios.append(check_field(_np(out0), ref, e[0], what))
        elif out_mode == ao.OUT_INTENSITY:
            ratios.append(check_field(_np(out0), np.abs(ref) ** 2, e[0], what))
            if with_out1:
                ratios.append(check_field(_np(out1), ref, e[1], what + " out1"))
        else:
            ratios.append(check_field(polar(_np(out0), _np(out1)), ref, polar(e[0], e[1]), what))
    return ratios


@pytest.mark.parametrize("n,pad,optics", CASES, ids=[f"{n}{'p' if p else ''}-{o}" for n, p, o in CASES])
def test_mode_matrix(pkg, n, pad, optics):
    L = pkg._lib
    lamb, px = OPTICS[optics]
    m = 2 * n if pad else n
    b, c = (1, 2) if m >= 2048 else (2, 3)
    off = 1 if (optics == "ring" and m in (1024, 2048)) else 0
    rng = np.random.default_rng(1000 * n + 10 * pad + (optics == "ring"))
    shape = (b, c, n, n)
    ratios, gz = [], []
    print(f"\nN={n} pad={pad} {optics} B={b} C={c} buffer offset {off}")
    for i, in_mode in enumerate(IN_MODES):
        z = rng.uniform(-20e-3, 20e-3, b).astype(np.float64 if (i + (optics == "ring")) % 2 else np.float32)
        zt = torch.from_numpy(z).cuda()
        in0, in1 = random_inputs(in_mode, shape, rng, IN_SCALE)
        o = ao.input_field(in_mode, in0, in1, IN_SCALE)
        ref, dudz = ao.asm_dudz(o, lamb, z, px, pad)
        c64 = ao.asm_c64(o, lamb, z, px, pad)
        # the constant amplitude is one device scalar; every other buffer carries the case's offset
        inp = (to_device(in0, 0 if in_mode == ao.IN_CONST_AMP_PHASE else off), to_device(in1, off))
        ratios += _check_forward(L, inp, zt, ref, c64, b, c, n, pad, in_mode, lamb, px, off)
        # distance gradient, both cotangents; the intensity one takes the forward field U (complex64) it belongs to
        for cot_mode in (ao.IN_COMPLEX, ao.IN_COT_FIELD):
            if cot_mode == ao.IN_COMPLEX:
                g = (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)
                cot, kshift = (to_device(g, off), None), 0.0
            else:
                w = rng.uniform(-1.0, 1.0, shape).astype(np.float32)
                u = ref.astype(np.complex64)
                g = 2.0 * w.astype(np.float64) * u
                cot, kshift = (to_device(w, off), to_device(u, off)), 1.0
            want, scale = ao.grad_z_sum(g, ref, dudz, lamb, z, kshift)
            got = torch.empty(b, dtype=torch.float64, device="cuda")
            abi_grad_z(L, inp[0], inp[1], zt, cot[0], cot[1], cot_mode, got, b, c, n, pad, in_mode, lamb, px, IN_SCALE)
            torch.cuda.synchronize()
            gz.append(check_grad_z(_np(got), want, scale, f"in{in_mode} cot{cot_mode} {z.dtype}"))
    # adjoint: g or 2 w U in, grad_O or (dL/dA, dL/dphase) out
    for j, in_mode in enumerate((ao.IN_COMPLEX, ao.IN_COT_FIELD)):
        z = rng.uniform(-20e-3, 20e-3, b).astype(np.float32 if (j + (optics == "ring")) % 2 else np.float64)
        zt = torch.from_numpy(z).cuda()
        in0, in1 = random_inputs(in_mode, shape, rng)
        gfield = ao.input_field(in_mode, in0, in1)
        ref = ao.asm_c128(gfield, lamb, z, px, pad, adjoint=True)
        c64 = ao.asm_c64(gfield, lamb, z, px, pad, adjoint=True)
        inp = (to_device(in0, off), to_device(in1, off))
        out0 = empty_device(shape, torch.complex64, off)
        abi_adjoint(L, inp[0], inp[1], zt, None, None, out0, None, b, c, n, pad, in_mode, ao.OUT_COMPLEX, lamb, px)
        torch.cuda.synchronize()
        ratios.append(check_field(_np(out0), ref, c64, f"adj in{in_mode} out{ao.OUT_COMPLEX} {z.dtype}"))
        amp, ph = random_inputs(ao.IN_AMP_PHASE, shape, rng, IN_SCALE)
        ga, gp = empty_device(shape, torch.float32, off), empty_device(shape, torch.float32, off)
        abi_adjoint(L, inp[0], inp[1], zt, to_device(amp, off), to_device(ph, off), ga, gp, b, c, n, pad, in_mode,
                    ao.OUT_GRAD_AP, lamb, px, IN_SCALE)
        torch.cuda.synchronize()
        r, e = ao.grad_ap(ref, amp, ph, IN_SCALE), ao.grad_ap(c64, amp, ph, IN_SCALE)
        ratios.append(check_field(_np(ga), r[0], e[0], f"adj in{in_mode} GRAD_AP dA"))
        ratios.append(check_field(_np(gp), r[1], e[1], f"adj in{in_mode} GRAD_AP dphase"))
    print(f"N={n} pad={pad} {optics}: worst kernel / c64 ratio {max(ratios):.2f} (KCAL {KCAL}), "
          f"worst grad_z |d|/S {max(gz):.2e}")
