"""CPU: the bounds of the band-limit GPU tests see a wrong band limit.  Each planted defect, applied to the oracle, is
rejected by the helper the GPU test uses for it (per-bin TOL_H, field KCAL, grad_z TOL_GZ), and a correct complex64
pipeline with the right mask passes the same helpers.  Samples carry distances whose limits are about M/4 and M/3."""
import numpy as np
import pytest

from oracle import asm_oracle as ao
import _band_limit as bl
from _parity import OPTICS, check_field, check_grad_z, check_transfer, recover_h

LAMB, PX = OPTICS["default"]


def _z(m, dtype=np.float32):
    return np.array([bl.z_for_lim(m, LAMB, PX, m // 4), bl.z_for_lim(m, LAMB, PX, m // 3)], dtype=dtype)


def _masked(h, keep):
    return np.where(keep, h, 0.0)


def _defect_h(defect, m, n, d):
    """[B, M, M] band-limited transfer function (n: the field size, m = n or 2n) with one planted defect (or none)."""
    h = ao.transfer_function(m, n, LAMB, PX, d)
    lim, keep = bl.band_limit_mask(m, LAMB, PX, d)
    k = np.arange(m)
    k = np.abs(np.where(k < m / 2, k, k - m))
    if defect == "lim_plus_one":
        ok = k[None, :] <= lim[:, None] + 1
        keep = ok[:, :, None] & ok[:, None, :]
    elif defect == "lim_minus_one":
        ok = k[None, :] <= lim[:, None] - 1
        keep = ok[:, :, None] & ok[:, None, :]
    elif defect == "one_axis":
        keep = np.broadcast_to((k[None, :] <= lim[:, None])[:, :, None], keep.shape)
    elif defect == "circular":
        keep = k[None, :, None] ** 2 + k[None, None, :] ** 2 <= lim[:, None, None] ** 2
    elif defect == "df_from_n":          # the window S = N px instead of M px: the limit of an FFT of size N
        ok = k[None, :] <= bl.band_limit_mask(n, LAMB, PX, d)[0][:, None]
        keep = ok[:, :, None] & ok[:, None, :]
    elif defect == "neighbour_z":
        _, keep = bl.band_limit_mask(m, LAMB, PX, np.roll(d, 1))
    elif defect == "no_mask":
        return h
    return _masked(h, keep)


H_DEFECTS = ["lim_plus_one", "lim_minus_one", "one_axis", "circular", "neighbour_z", "no_mask"]


@pytest.mark.parametrize("m", [32, 64, 256, 45])
@pytest.mark.parametrize("defect", [None] + H_DEFECTS)
def test_per_bin_bound_sees_the_mask(m, defect):
    """Impulse response -> recovered H, per-bin TOL_H: forward (H mask) and adjoint (conj(H) mask)."""
    d = _z(m)
    ref = _masked(ao.transfer_function(m, m, LAMB, PX, d), bl.band_limit_mask(m, LAMB, PX, d)[1])[:, None]
    imp = np.zeros((2, 2, m, m), dtype=np.complex64)
    imp[:, :, 0, 0] = 1.0
    for adjoint in (False, True):
        want = np.conj(ref) if adjoint else ref
        if defect is None:
            check_transfer(recover_h(bl.propagate(imp, LAMB, d, PX, adjoint=adjoint, dtype=np.complex64)), want, "c64")
            continue
        h = _defect_h(defect, m, m, d)[:, None]
        u = ao.propagate_h(imp, h, adjoint=adjoint, dtype=np.complex64)
        with pytest.raises(AssertionError):
            check_transfer(recover_h(u), want, f"{defect} adjoint={adjoint}")


@pytest.mark.parametrize("m,pad", [(64, False), (64, True), (256, False), (128, True)])
@pytest.mark.parametrize("defect", [None, "lim_plus_one", "one_axis", "circular", "df_from_n", "neighbour_z",
                                    "adjoint_unmasked"])
def test_field_bound_sees_the_mask(m, pad, defect):
    """White random fields, rel-L2 <= KCAL x (complex64 pipeline's error): forward and adjoint."""
    n = m // 2 if pad else m
    if defect == "df_from_n" and not pad:
        pytest.skip("df from N differs from df from M only with padding")
    rng = np.random.default_rng(m + pad)
    o = (rng.standard_normal((2, 2, n, n)) + 1j * rng.standard_normal((2, 2, n, n))).astype(np.complex64)
    d = _z(m)
    for adjoint in (False, True):
        ref = bl.propagate(o, LAMB, d, PX, pad, adjoint)
        c64 = bl.propagate(o, LAMB, d, PX, pad, adjoint, dtype=np.complex64)
        if defect is None:
            check_field(c64, ref, c64, f"c64 adjoint={adjoint}")
            continue
        if defect == "adjoint_unmasked":
            if not adjoint:
                continue
            h = _defect_h("no_mask", m, n, d)
        else:
            h = _defect_h(defect, m, n, d)
        bad = ao.propagate_h(o, h[:, None], pad, adjoint, dtype=np.complex64)
        with pytest.raises(AssertionError):
            check_field(bad, ref, c64, f"{defect} adjoint={adjoint}")


def _grad_z_c64(o, g, d, pad, kshift, deriv_mask):
    """Re sum conj(g) dU/dz in a complex64 pipeline; the derivative filter i K (kz - kshift / lambda) H, masked or not."""
    import scipy.fft as sf
    n = o.shape[-1]
    m = bl.fft_size(n, pad)
    p = (m - n) // 2
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    x = o.astype(np.complex64)[:, :, idx][:, :, :, idx]
    h = bl.h_bl(m, n, LAMB, PX, d, band_limit=deriv_mask)[:, None]
    filt = (1j * ao.grad_constant(d) * (ao.kz_unshifted(m, n, LAMB, PX) - kshift / LAMB) * h).astype(np.complex64)
    du = sf.ifft2(filt * sf.fft2(x))[:, :, p:p + n, p:p + n]
    return np.real(np.conj(g.astype(np.complex64)) * du).astype(np.float64).sum(axis=(1, 2, 3))


@pytest.mark.parametrize("m,pad", [(64, False), (128, True)])
@pytest.mark.parametrize("cot", ["complex", "intensity"])
@pytest.mark.parametrize("defect", [None, "deriv_unmasked"])
def test_grad_z_bound_sees_the_mask(m, pad, cot, defect):
    n = m // 2 if pad else m
    rng = np.random.default_rng(9)
    o = (rng.standard_normal((2, 2, n, n)) + 1j * rng.standard_normal((2, 2, n, n))).astype(np.complex64)
    d = _z(m)
    u, du = bl.dudz(o, LAMB, d, PX, pad)
    if cot == "complex":
        g, kshift = rng.standard_normal(o.shape) + 1j * rng.standard_normal(o.shape), 0.0
    else:
        g, kshift = 2.0 * rng.uniform(-1, 1, o.shape) * u.astype(np.complex64), 1.0
    ref, scale = ao.grad_z_sum(g, u, du, LAMB, d, kshift)
    if defect is None:
        check_grad_z(_grad_z_c64(o, g, d, pad, kshift, True), ref, scale, "c64")
        return
    with pytest.raises(AssertionError):
        check_grad_z(_grad_z_c64(o, g, d, pad, kshift, False), ref, scale, defect)
