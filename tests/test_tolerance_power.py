"""CPU: the bounds of the GPU parity tests discriminate.  Each planted defect -- one bin, one row, one rounded constant,
one folded edge, one channel's distance, one derivative bin -- fails the helper it targets, and the correct complex64
pipeline (oracle.asm_oracle.asm_c64) passes the same helper.  Ring optics (a ring of evanescent bins), small sizes."""
import numpy as np
import pytest

from oracle import asm_oracle as ao
from _parity import OPTICS, check_field, check_grad_z, check_transfer, recover_h

LAMB, PX = OPTICS["ring"]
Z32 = np.array([6e-3, -20e-3], dtype=np.float32)
Z64 = np.array([0.0123456789, 0.5], dtype=np.float64)


def _kz(m, n):
    return ao.kz_unshifted(m, n, LAMB, PX)


def _h_from(kz, c):
    return np.exp(1j * (np.asarray(c, dtype=np.float64)[:, None, None] * kz[None]))


def _defect_h(defect, m, n, d):
    """[B, M, M] transfer function with one planted defect (or none)."""
    kz = _kz(m, n)
    c = ao.phase_constant(d)
    if defect == "kappa_fp32":
        kz = (kz / (2 * np.pi)).astype(np.float32).astype(np.float64) * (2 * np.pi)
    if defect == "phase_constant_fp32":
        c = ao.phase_constant(np.asarray(d, dtype=np.float32))
    h = _h_from(kz, c)
    if defect == "one_bin_1e-3":
        h[:, 3, 5] *= np.exp(1e-3j)
    if defect == "one_bin_0.1":
        h[:, 3, 5] *= np.exp(0.1j)
    if defect == "nyquist_row_conj":
        h[:, m // 2, :] = np.conj(h[:, m // 2, :])
    if defect == "evanescent_zero":
        h[:, kz == 0] = 0.0
    return h


def _fields(m, pad):
    n = m // 2 if pad else m
    rng = np.random.default_rng(m + pad)
    o = (rng.standard_normal((2, 2, n, n)) + 1j * rng.standard_normal((2, 2, n, n))).astype(np.complex64)
    return n, o


def _wrong_channel_h(h, c):
    """[B, C, M, M]: channel 1 of every sample propagated with the next sample's distance."""
    hh = np.repeat(h[:, None], c, axis=1)
    hh[:, 1] = np.roll(h, -1, axis=0)
    return hh


H_DEFECTS = ["one_bin_1e-3", "nyquist_row_conj", "evanescent_zero", "kappa_fp32", "phase_constant_fp32", "wrong_channel_z"]


@pytest.mark.parametrize("m", [32, 64, 256])
@pytest.mark.parametrize("defect", [None] + H_DEFECTS)
def test_per_bin_bound(m, defect):
    """Impulse response -> recovered H, bound TOL_H per bin (transfer-function tests)."""
    d = Z64 if defect == "phase_constant_fp32" else Z32
    imp = np.zeros((2, 2, m, m), dtype=np.complex64)
    imp[:, :, 0, 0] = 1.0
    ref = _h_from(_kz(m, m), ao.phase_constant(d))[:, None]
    if defect is None:   # the complex64 pipeline is accepted
        u = ao.asm_c64(imp, LAMB, d, PX)
        check_transfer(recover_h(u), ref, "c64")
        return
    h = _defect_h(None if defect == "wrong_channel_z" else defect, m, m, d)
    hh = _wrong_channel_h(h, 2) if defect == "wrong_channel_z" else h[:, None]
    u = ao.propagate_h(imp, hh, dtype=np.complex64)
    with pytest.raises(AssertionError):
        check_transfer(recover_h(u), ref, defect)


FIELD_DEFECTS = ["one_bin_0.1", "nyquist_row_conj", "evanescent_zero", "kappa_fp32", "phase_constant_fp32",
                 "adjoint_fold_dropped", "wrong_channel_z"]


def _fold_dropped(y, n, p):
    """replicate_pad_T without the fold of the last p columns onto column n-1."""
    z = ao.replicate_pad_T(y, n, p)
    z[:, :, :, n - 1] -= y[:, :, p:p + n, p + n:].sum(axis=3)
    z[:, :, n - 1, n - 1] -= y[:, :, p + n:, p + n:].sum(axis=(2, 3))
    return z


@pytest.mark.parametrize("m,pad", [(64, False), (64, True), (256, False), (128, True)])
@pytest.mark.parametrize("defect", [None] + FIELD_DEFECTS)
def test_field_bound(m, pad, defect):
    """White random fields, rel-L2 bound KCAL x (complex64 pipeline's error) (mode-matrix tests)."""
    n, o = _fields(m, pad)
    adjoint = defect == "adjoint_fold_dropped" or (defect is None and pad)
    if defect == "adjoint_fold_dropped" and not pad:
        pytest.skip("the fold exists only with padding")
    d = Z64 if defect == "phase_constant_fp32" else Z32
    ref = ao.asm_c128(o, LAMB, d, PX, pad, adjoint=adjoint)
    c64 = ao.asm_c64(o, LAMB, d, PX, pad, adjoint=adjoint)
    if defect is None:
        check_field(c64, ref, c64, "c64")
        check_field(ao.asm_c64(o, LAMB, d, PX, pad), ao.asm_c128(o, LAMB, d, PX, pad), ao.asm_c64(o, LAMB, d, PX, pad), "c64 fwd")
        return
    if defect == "adjoint_fold_dropped":
        h = _defect_h(None, m, n, d)[:, None].astype(np.complex64)
        mm, p = m, (m - n) // 2
        x = np.zeros((2, 2, mm, mm), dtype=np.complex64)
        x[:, :, p:p + n, p:p + n] = o
        import scipy.fft as sf
        bad = _fold_dropped(sf.ifft2(np.conj(h) * sf.fft2(x)), n, p)
    else:
        h = _defect_h(None if defect == "wrong_channel_z" else defect, m, n, d)
        hh = _wrong_channel_h(h, 2) if defect == "wrong_channel_z" else h[:, None]
        bad = ao.propagate_h(o, hh, pad, dtype=np.complex64)
    with pytest.raises(AssertionError):
        check_field(bad, ref, c64, defect)


def _grad_z_defect(o, g, d, pad, kshift, neighbour):
    """Re sum conj(g) dU/dz with dU/dz evaluated from kz rolled by one bin along the columns if ``neighbour``."""
    n = o.shape[-1]
    m = 2 * n if pad else n
    p = (m - n) // 2
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    x = o.astype(np.complex64)[:, :, idx][:, :, :, idx]
    kz = _kz(m, n)
    kd = np.roll(kz, 1, axis=1) if neighbour else kz
    h = _h_from(kz, ao.phase_constant(d))[:, None].astype(np.complex64)
    filt = (1j * ao.grad_constant(d) * (kd - kshift / LAMB)).astype(np.complex64)
    import scipy.fft as sf
    du = sf.ifft2(filt * h * sf.fft2(x))[:, :, p:p + n, p:p + n]
    return np.real(np.conj(g.astype(np.complex64)) * du).astype(np.float64).sum(axis=(1, 2, 3))


@pytest.mark.parametrize("m,pad", [(64, False), (128, True)])
@pytest.mark.parametrize("cot", ["complex", "intensity"])
@pytest.mark.parametrize("defect", [None, "neighbour_kz"])
def test_grad_z_bound(m, pad, cot, defect):
    """grad_z: |delta| <= TOL_GZ * S_b; a complex64 evaluation passes, a derivative from the neighbouring bin's kz fails."""
    n, o = _fields(m, pad)
    d = Z32
    rng = np.random.default_rng(9)
    if cot == "complex":
        g, kshift = (rng.standard_normal(o.shape) + 1j * rng.standard_normal(o.shape)), 0.0
    else:
        u = ao.asm_c128(o, LAMB, d, PX, pad).astype(np.complex64)
        g, kshift = 2.0 * rng.uniform(-1, 1, o.shape) * u, 1.0
    ref, scale = ao.asm_grad_z(o, g, LAMB, d, PX, pad, kshift=kshift)
    if defect is None:
        check_grad_z(_grad_z_defect(o, g, d, pad, kshift, False), ref, scale, "c64")
        return
    bad = _grad_z_defect(o, g, d, pad, kshift, True)
    with pytest.raises(AssertionError):
        check_grad_z(bad, ref, scale, defect)


def test_transfer_function_matches_asm():
    """transfer_function / propagate_h / asm_c128 restate asm_closed_form and asm_adjoint exactly."""
    rng = np.random.default_rng(0)
    for n, pad in ((64, False), (32, True), (45, False)):
        o = rng.standard_normal((2, 1, n, n)) + 1j * rng.standard_normal((2, 1, n, n))
        d = np.array([1e-3, -3e-3], dtype=np.float32)
        assert ao.rel_l2(ao.asm_c128(o, LAMB, d, PX, pad), ao.asm_closed_form(o, LAMB, d, PX, pad)) < 1e-13
        assert ao.rel_l2(ao.asm_c128(o, LAMB, d, PX, pad, adjoint=True), ao.asm_adjoint(o, LAMB, d, PX, pad)) < 1e-13
        assert ao.rel_l2(ao.asm_c128(o, LAMB, d, PX, pad), ao.asm(o, LAMB, d, PX, pad)) < 1e-12
        g = rng.standard_normal(o.shape) + 1j * rng.standard_normal(o.shape)
        gd, s = ao.asm_grad_z(o, g, LAMB, d, PX, pad)
        assert np.allclose(gd, ao.asm_grad_d(o, g, LAMB, d, PX, pad), rtol=1e-12, atol=0) and np.all(s >= np.abs(gd))
        # the shifted derivative gives the same gradient for the intensity cotangent g = 2 w U
        u = ao.asm_c128(o, LAMB, d, PX, pad)
        w = rng.uniform(-1, 1, o.shape)
        g0, _ = ao.asm_grad_z(o, 2 * w * u, LAMB, d, PX, pad)
        g1, s1 = ao.asm_grad_z(o, 2 * w * u, LAMB, d, PX, pad, kshift=1.0)
        assert np.all(np.abs(g0 - g1) <= 1e-9 * s1)


def test_input_modes_and_grad_constant():
    rng = np.random.default_rng(1)
    ph = rng.uniform(-1e5, 1e5, (1, 1, 4, 4)).astype(np.float32)
    a = rng.uniform(0, 1, ph.shape).astype(np.float32)
    e = np.exp(1j * (ph * np.float32(0.7)).astype(np.float32).astype(np.float64))
    assert np.array_equal(ao.input_field(ao.IN_AMP_PHASE, a, ph, 0.7), a.astype(np.float64) * e)
    assert np.array_equal(ao.input_field(ao.IN_CONST_AMP_PHASE, np.float32([0.6]), ph, 0.7), float(np.float32(0.6)) * e)
    u = (rng.standard_normal(ph.shape) + 1j * rng.standard_normal(ph.shape)).astype(np.complex64)
    assert np.array_equal(ao.input_field(ao.IN_COT_FIELD, a, u), 2.0 * a.astype(np.float64) * u.astype(np.complex128))
    assert np.array_equal(ao.input_field(ao.IN_SQRT_REAL, a), np.sqrt(a.astype(np.float64)) + 0j)
    assert ao.grad_constant(np.float32(1e-3)) == float(np.float32(2 * np.pi))
    assert ao.grad_constant(np.float64(1e-3)) == 2 * np.pi
