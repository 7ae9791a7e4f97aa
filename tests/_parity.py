"""Assertion helpers and C-ABI call wrappers shared by the transfer-function, mode-matrix and tolerance-power tests.

The bounds are calibrated on a correct single-precision pipeline (``asm_oracle.asm_c64``):
  - per-bin transfer function: max |H_kernel - H_oracle| <= tol_h(M) (TOL_H for the FFT sizes; the complex64
    pipeline stays below 7.4e-7);
  - fields: rel-L2(kernel, float64) <= KCAL * rel-L2(complex64 pipeline, float64), per output;
  - distance gradients: |grad - oracle| <= TOL_GZ * S_b, S_b = sum |Re(conj(g) dU/dz)| (the rounding scale of the sum).
``tests/test_tolerance_power.py`` checks on the CPU that each bound rejects planted one-bin, one-row and one-constant
defects while accepting the complex64 pipeline.
"""
from __future__ import annotations

import ctypes

import numpy as np

from oracle import asm_oracle as ao

TOL_H = 1e-5
KCAL = 8.0
TOL_GZ = 1e-5

# (wavelength, pixel size): no bin evanescent / a ring of evanescent bins / most bins evanescent
OPTICS = {"default": (532e-9, 1.5e-6), "ring": (532e-9, 0.3e-6), "evanescent": (633e-9, 0.2e-6)}


def evanescent_fraction(m: int, n: int, lamb: float, px: float) -> float:
    k = np.arange(m, dtype=np.float64)
    k = np.where(k < m / 2, k, k - m)
    f = (k / 2) / (n * px) if m == 2 * n else k / (n * px)
    arg = 1.0 - lamb ** 2 * (f[:, None] ** 2 + f[None, :] ** 2)
    return float(np.mean(arg <= 0))


def assert_well_conditioned(m: int, n: int, lamb: float, px: float, zmax: float) -> float:
    """Near the evanescent circle kz = sqrt(arg) / lamb is ill-conditioned (arg = 1 - s^2 (ku^2 + kv^2)); the kernel and
    the oracle may round arg differently by one unit of 2^-53.  Require that this moves no bin's phase by more than
    1e-6 rad at |z| <= zmax, so that a per-bin difference above TOL_H is a defect and not a formulation difference.
    Returns the worst phase change."""
    s2 = (lamb / (m * px)) ** 2
    k = np.arange(m, dtype=np.float64)
    k = np.where(k < m / 2, k, k - m)
    arg = 1.0 - s2 * (k[:, None] ** 2 + k[None, :] ** 2)
    a = np.abs(arg)
    assert a.min() > 1e-12, "a bin lies on the evanescent circle: kernel and oracle may clamp it differently"
    pos = arg[arg > 0]
    worst = 2 * np.pi * zmax / lamb * 0.5 * 2.0 ** -53 / np.sqrt(pos.min())
    assert worst <= 1e-6, worst
    return float(worst)


def recover_h(u: np.ndarray) -> np.ndarray:
    """The kernel's transfer function from its response to a unit impulse at (0, 0): float64 fft2 of the output."""
    import scipy.fft as sf
    return sf.fft2(np.asarray(u).astype(np.complex128), axes=(-2, -1), workers=-1)


def tol_h(m: int) -> float:
    """Per-bin bound at transform size m.  The FFT families round like log m and stay near 1e-6 up to 4096 on a B200.
    The matrix-product path (m not a power of two) sums m fp32 products per output serially, so its rounding grows like
    sqrt(m): measured 0.7e-6 at 45, 2.6e-6 at 250, up to 1.3e-5 at 1000 with 69 % evanescent bins."""
    return TOL_H if m & (m - 1) == 0 else TOL_H * max(1.0, float(np.sqrt(m / 128)))


def check_transfer(h_kernel: np.ndarray, h_oracle: np.ndarray, what: str = "") -> float:
    tol = tol_h(h_oracle.shape[-1])
    err = float(np.max(np.abs(h_kernel - h_oracle)))
    print(f"  H {what}: max |dH| = {err:.3e}  (bound {tol:.1e})")
    assert err <= tol, (what, err)
    return err


def _as_complex(x):
    return np.asarray(x).astype(np.complex128)


def field_errors(kernel: np.ndarray, oracle: np.ndarray, c64: np.ndarray):
    """(kernel error, complex64-pipeline error), rel-L2 against the float64 oracle."""
    return ao.rel_l2(_as_complex(kernel), _as_complex(oracle)), ao.rel_l2(_as_complex(c64), _as_complex(oracle))


def check_field(kernel, oracle, c64, what: str = "") -> float:
    """rel-L2(kernel) <= KCAL * rel-L2(c64).  Returns the ratio."""
    ek, ec = field_errors(kernel, oracle, c64)
    ec = max(ec, 1e-9)
    print(f"  {what}: err {ek:.3e}  bound {KCAL * ec:.3e}  (c64 {ec:.3e}, ratio {ek / ec:.2f})")
    assert ek <= KCAL * ec, (what, ek, ec)
    return ek / ec


def polar(a, ang):
    """|U| e^{i angle}: angles are compared through the field they describe, never raw (the branch cut at +-pi)."""
    return np.asarray(a, dtype=np.float64) * np.exp(1j * np.asarray(ang, dtype=np.float64))


def check_grad_z(kernel, oracle, scale, what: str = "") -> float:
    """|kernel - oracle| <= TOL_GZ * S_b per sample.  Returns the worst |delta| / S_b."""
    kernel, oracle, scale = (np.asarray(v, dtype=np.float64).reshape(-1) for v in (kernel, oracle, scale))
    rel = np.abs(kernel - oracle) / scale
    print(f"  grad_z {what}: max |d|/S = {rel.max():.3e}  (bound {TOL_GZ:.1e})")
    assert np.all(rel <= TOL_GZ), (what, rel.tolist())
    return float(rel.max())


# --------------------------------------------------------------------------------------------
# inputs of every in_mode
# --------------------------------------------------------------------------------------------
WIDE_PHASE = (4.9e4, 5.1e4)   # |phase * in_scale| on both sides of sincos_reduced's switch to the library sincosf


def random_inputs(in_mode: int, shape, rng, in_scale: float = 0.7, wide_rows: int = 2):
    """White random (in0, in1) for ``in_mode`` (fp32 / complex64).  Phases of the first ``wide_rows`` rows of every plane
    have |phase * in_scale| in WIDE_PHASE, with both signs."""
    n = shape[-1]

    def cplx():
        return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)

    def phase():
        ph = rng.uniform(-np.pi, np.pi, shape)
        if wide_rows:
            w = rng.uniform(*WIDE_PHASE, shape[:-2] + (wide_rows, n)) * rng.choice([-1.0, 1.0], shape[:-2] + (wide_rows, n))
            ph[..., :wide_rows, :] = w / in_scale
        return ph.astype(np.float32)

    if in_mode == ao.IN_COMPLEX:
        return cplx(), None
    if in_mode == ao.IN_AMP_PHASE:
        return rng.uniform(0.2, 1.5, shape).astype(np.float32), phase()
    if in_mode == ao.IN_CONST_AMP_PHASE:
        return np.array([0.6], dtype=np.float32), phase()
    if in_mode == ao.IN_SQRT_REAL:
        return rng.uniform(0.0, 2.0, shape).astype(np.float32), None
    if in_mode == ao.IN_COT_FIELD:
        return rng.uniform(-1.0, 1.0, shape).astype(np.float32), cplx()
    if in_mode == ao.IN_REAL:
        return rng.standard_normal(shape).astype(np.float32), None
    raise ValueError(in_mode)


# --------------------------------------------------------------------------------------------
# C ABI through ctypes (GPU tests only)
# --------------------------------------------------------------------------------------------
def to_device(a, offset: int = 0):
    """numpy -> CUDA tensor stored ``offset`` elements into a fresh allocation (offset 1 breaks 16-byte alignment)."""
    import torch
    if a is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(a))
    flat = torch.empty(t.numel() + offset, dtype=t.dtype, device="cuda")
    v = flat[offset:].view(t.shape)
    v.copy_(t)
    return v


def empty_device(shape, dtype, offset: int = 0):
    import torch
    n = int(np.prod(shape))
    return torch.empty(n + offset, dtype=dtype, device="cuda")[offset:].view(tuple(shape))


def _ptr(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _workspace(lib, b, c, n, pad):
    import torch
    return torch.empty(lib.asm_b200_workspace_bytes(b, c, n, int(pad)), dtype=torch.uint8, device="cuda")


def _zdtype(L, z):
    import torch
    return L.Z_F64 if z.dtype == torch.float64 else L.Z_F32


def abi_forward(L, in0, in1, z, out0, out1, b, c, n, pad, in_mode, out_mode, lamb, px, in_scale=1.0, out_scale=1.0):
    lib = L.load()
    ws = _workspace(lib, b, c, n, pad)
    L.check(lib.asm_b200_forward(_ptr(in0), _ptr(in1), _ptr(z), _zdtype(L, z), _ptr(out0), _ptr(out1), b, c, n, int(pad),
                                 in_mode, out_mode, lamb, px, in_scale, out_scale, _ptr(ws), ws.numel(), _stream()))


def abi_adjoint(L, in0, in1, z, aux0, aux1, out0, out1, b, c, n, pad, in_mode, out_mode, lamb, px, in_scale=1.0):
    lib = L.load()
    ws = _workspace(lib, b, c, n, pad)
    L.check(lib.asm_b200_adjoint(_ptr(in0), _ptr(in1), _ptr(z), _zdtype(L, z), _ptr(aux0), _ptr(aux1), _ptr(out0),
                                 _ptr(out1), b, c, n, int(pad), in_mode, out_mode, lamb, px, in_scale, _ptr(ws), ws.numel(),
                                 _stream()))


def abi_grad_z(L, in0, in1, z, cot0, cot1, cot_mode, grad, b, c, n, pad, in_mode, lamb, px, in_scale=1.0):
    lib = L.load()
    ws = _workspace(lib, b, c, n, pad)
    L.check(lib.asm_b200_grad_z(_ptr(in0), _ptr(in1), _ptr(z), _zdtype(L, z), _ptr(cot0), _ptr(cot1), cot_mode,
                                _ptr(grad), b, c, n, int(pad), in_mode, lamb, px, in_scale, _ptr(ws), ws.numel(), _stream()))
