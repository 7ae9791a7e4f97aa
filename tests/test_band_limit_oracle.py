"""CPU: the band-limited oracle (``band_limit_mask`` and the operators of tests/_band_limit.py).

  - where the limit keeps every bin (lim >= M/2) the band-limited operator is the plain one, bit for bit;
  - the mask equals an independent restatement |f_x|, |f_y| <= f_lim(z), f = k df, on seeded (M, px, lambda, z) draws;
  - the adjoint is the adjoint (<A x, y> = <x, A^H y>), padded and unpadded;
  - grad_z is the derivative (central difference away from a jump of lim);
  - against a direct first-kind Rayleigh-Sommerfeld sum the band limit removes most of the aliasing error at long
    distances and costs accuracy at short ones (why it is opt-in).
"""
import numpy as np
import pytest

from oracle import asm_oracle as ao
import _band_limit as bl

LAMB, PX = 532e-9, 1.5e-6


def _field(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


@pytest.mark.parametrize("n,pad", [(64, False), (32, True), (45, False), (256, False)])
def test_full_band_equals_plain_bit_for_bit(n, pad):
    m = bl.fft_size(n, pad)
    z = np.array([1e-5, -2e-5], dtype=np.float32)          # short distances: lim clamps at M
    lim, keep = bl.band_limit_mask(m, LAMB, PX, z)
    assert np.all(lim >= m // 2) and keep.all()
    o = _field((2, 2, n, n), n)
    for adjoint in (False, True):
        a = bl.propagate(o, LAMB, z, PX, pad, adjoint, band_limit=True)
        b = bl.propagate(o, LAMB, z, PX, pad, adjoint, band_limit=False)
        assert np.array_equal(a, b)
    assert np.array_equal(bl.dudz(o, LAMB, z, PX, pad, True)[1], bl.dudz(o, LAMB, z, PX, pad, False)[1])


def test_mask_matches_independent_restatement():
    rng = np.random.default_rng(12)
    checked = rejected = 0
    while checked < 200:
        m = int(rng.choice([32, 45, 64, 92, 128, 250, 256, 1000, 1024, 2048, 4096]))
        px = float(rng.uniform(0.2e-6, 6e-6))
        lamb = float(rng.uniform(400e-9, 1100e-9))
        z = rng.uniform(-0.2, 0.2) * 10.0 ** rng.uniform(-4, 0)
        z = np.float32(z) if rng.random() < 0.5 else np.float64(z)
        if bl.lim_margin(m, lamb, px, z) < 1e-9:          # within rounding of a jump of lim: the two forms may disagree
            rejected += 1
            continue
        lim, keep = bl.band_limit_mask(m, lamb, px, z)
        df = 1.0 / (m * px)
        f_lim = 1.0 / (lamb * np.sqrt(1.0 + (2.0 * float(z) * df) ** 2))
        k = np.arange(m)
        f = np.where(k < (m + 1) // 2, k, k - m) * df
        ok = np.abs(f) <= f_lim
        assert np.array_equal(keep[0], ok[:, None] & ok[None, :]), (m, px, lamb, z, lim)
        checked += 1
    assert rejected < 20


def test_lim_clamps_and_nan():
    lim, keep = bl.band_limit_mask(64, LAMB, 100.0, np.array([0.0, np.nan, np.inf]))
    assert lim.tolist() == [64, 64, 0]                       # S / lambda >> INT_MAX clamps; NaN keeps all; inf keeps DC
    assert keep[0].all() and keep[1].all() and keep[2].sum() == 1 and keep[2, 0, 0]


@pytest.mark.parametrize("n,pad", [(64, False), (32, True), (45, False), (46, True)])
def test_adjoint_identity(n, pad):
    m = bl.fft_size(n, pad)
    z = np.array([bl.z_for_lim(m, LAMB, PX, m // 4), bl.z_for_lim(m, LAMB, PX, m // 3)], dtype=np.float64)
    x, y = _field((2, 2, n, n), 1), _field((2, 2, n, n), 2)
    ax = bl.propagate(x, LAMB, z, PX, pad)
    ahy = bl.propagate(y, LAMB, z, PX, pad, adjoint=True)
    lhs, rhs = np.vdot(y, ax), np.vdot(ahy, x)
    assert abs(lhs - rhs) <= 1e-12 * abs(lhs), (lhs, rhs)
    # the mask bites: the band-limited field is not the plain one
    assert ao.rel_l2(ax, bl.propagate(x, LAMB, z, PX, pad, band_limit=False)) > 1e-2


@pytest.mark.parametrize("n,pad", [(64, False), (32, True)])
def test_grad_z_is_the_derivative_between_jumps(n, pad):
    m = bl.fft_size(n, pad)
    z0 = bl.z_for_lim(m, LAMB, PX, m // 4)
    eps = 1e-10                                                       # k eps ~ 1e-3: the carrier e^{i k z} is resolved
    assert bl.lim_margin(m, LAMB, PX, [z0 - eps, z0 + eps]) > 1e-3   # no jump of lim inside the difference
    o, g = _field((1, 2, n, n), 3), _field((1, 2, n, n), 4)
    u, du = bl.dudz(o, LAMB, np.float64(z0), PX, pad)
    grad, scale = ao.grad_z_sum(g, u, du, LAMB, np.array([z0]))
    up = bl.propagate(o, LAMB, np.float64(z0 + eps), PX, pad)
    um = bl.propagate(o, LAMB, np.float64(z0 - eps), PX, pad)
    fd = np.real(np.vdot(g, up - um)) / (2 * eps)
    assert abs(grad[0] - fd) <= 1e-6 * scale[0], (grad[0], fd, scale[0])


# --------------------------------------------------------------------------------------------
# against a direct first-kind Rayleigh-Sommerfeld sum: 64 x 64 object, padded (FFT 128), lambda 532 nm, px 1.5 um
# --------------------------------------------------------------------------------------------
RS_N = 64


def _rs_object():
    """Gaussian-apodised amplitude, smooth random phase (std 2 rad)."""
    rng = np.random.default_rng(0)
    y, x = np.mgrid[:RS_N, :RS_N] - (RS_N - 1) / 2
    amp = np.exp(-(x ** 2 + y ** 2) / (2 * (RS_N / 8) ** 2))
    f = np.fft.fftfreq(RS_N)
    smooth = np.exp(-(f[:, None] ** 2 + f[None, :] ** 2) / (2 * 0.05 ** 2))
    ph = np.real(np.fft.ifft2(np.fft.fft2(rng.standard_normal((RS_N, RS_N))) * smooth))
    ph *= 2 / ph.std()
    return amp * np.exp(1j * ph)


def _rayleigh_sommerfeld(o, z):
    """U(x) = sum_x' o(x') z / (2 pi r^2) (1 / r - i k) e^{i k r} px^2, r = |x - x'| with the plane distance z."""
    k = 2 * np.pi / LAMB
    xs = (np.arange(RS_N) - (RS_N - 1) / 2) * PX
    gx, gy = np.meshgrid(xs, xs, indexing="ij")
    gx, gy, ov = gx.ravel(), gy.ravel(), o.ravel()
    out = np.empty(RS_N * RS_N, dtype=np.complex128)
    for s in range(0, RS_N * RS_N, 512):
        dx = gx[s:s + 512, None] - gx[None]
        dy = gy[s:s + 512, None] - gy[None]
        r = np.sqrt(dx * dx + dy * dy + z * z)
        out[s:s + 512] = (z / (2 * np.pi * r * r) * (1 / r - 1j * k) * np.exp(1j * k * r)) @ ov * PX * PX
    return out.reshape(RS_N, RS_N)


# z: (max band-limited error, min plain error) -- observed 0.146 / 0.376 at 3 mm and 0.518 / 2.94 at 10 mm
RS_PINS = {3e-3: (0.16, 0.35), 10e-3: (0.55, 2.8)}


@pytest.mark.parametrize("z", [1e-3, 3e-3, 10e-3])
def test_band_limit_against_rayleigh_sommerfeld(z):
    o = _rs_object()
    ref = _rayleigh_sommerfeld(o, z)
    plain = bl.propagate(o[None, None], LAMB, np.float64(z), PX, True, band_limit=False)[0, 0]
    limited = bl.propagate(o[None, None], LAMB, np.float64(z), PX, True, band_limit=True)[0, 0]
    e_plain, e_bl = ao.rel_l2(plain, ref), ao.rel_l2(limited, ref)
    lim = int(bl.band_limit_mask(2 * RS_N, LAMB, PX, z)[0][0])
    print(f"z = {z * 1e3:.0f} mm: lim {lim} of {RS_N}, rel-L2 plain {e_plain:.3e}, band-limited {e_bl:.3e}")
    if z in RS_PINS:
        top_bl, bottom_plain = RS_PINS[z]
        assert e_bl < top_bl and e_plain > bottom_plain and e_bl < 0.45 * e_plain
    else:   # short distance: the limit cuts signal the plain spectrum samples correctly -- why it is opt-in
        assert e_plain < 2.5e-3 and e_bl > 2 * e_plain
