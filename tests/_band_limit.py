"""The band-limited angular spectrum on the host: ``band_limit_mask`` (the host's only statement of the rule) and the operators
built from it on top of oracle.asm_oracle, shared by the band-limit tests: H mask forward, conj(H) mask adjoint,
i K kz H mask for the distance derivative."""
from __future__ import annotations

import numpy as np

from oracle import asm_oracle as ao


def fft_size(n: int, pad: bool) -> int:
    return 2 * n if pad else n


def band_limit_mask(m: int, lamb: float, px: float, d):
    """(lim [len(d)] int64, mask [len(d), m, m] bool) of the band-limited angular spectrum (Matsushima & Shimobaba,
    Opt. Express 17, 19662, 2009), as the library evaluates it (include/asm_b200.h, asm_b200_*_bl):

        lim(z) = floor( S / (lamb sqrt(1 + q q)) ),  q = 2 z / S,  S = m px   (float64, this order; clamped to m)

    with z the float64 value of each distance (an fp32 distance converts exactly).  Bin (u, v) is kept iff
    |k(u)| <= lim and |k(v)| <= lim, k(u) = u < m/2 ? u : u - m as in ``asm_oracle.kz_unshifted``: |f_x|, |f_y| <=
    f_lim(z) = 1 / (lamb sqrt(1 + (2 z df)^2)), df = 1 / (m px).  ``m`` is the FFT size (n, or 2n padded).
    """
    z = np.atleast_1d(np.asarray(d)).astype(np.float64).reshape(-1)
    s = float(m) * float(px)
    q = (2.0 * z) / s
    lim = np.fmin(np.floor(s / (float(lamb) * np.sqrt(1.0 + q * q))), float(m)).astype(np.int64)
    k = np.arange(m, dtype=np.int64)
    k = np.abs(np.where(k < m / 2, k, k - m))
    keep = k[None, :] <= lim[:, None]
    return lim, keep[:, :, None] & keep[:, None, :]


def h_bl(m: int, n: int, lamb: float, px: float, d, band_limit: bool = True, lim_d=None) -> np.ndarray:
    """[len(d), m, m] transfer function, zeroed outside the band limit (``lim_d``: take the limit from these distances)."""
    h = ao.transfer_function(m, n, lamb, px, np.atleast_1d(d))
    if not band_limit:
        return h
    _, keep = band_limit_mask(m, lamb, px, np.atleast_1d(d) if lim_d is None else np.atleast_1d(lim_d))
    return np.where(keep, h, 0.0)


def propagate(o, lamb, d, px, pad=False, adjoint=False, band_limit=True, dtype=np.complex128):
    """The library's forward (or exact adjoint) operator with the band-limited H, in float64 or as a complex64 pipeline."""
    o = np.asarray(o)
    n = o.shape[-1]
    d = np.asarray(d).reshape(-1) if np.asarray(d).size == o.shape[0] else np.full(o.shape[0], d, dtype=np.asarray(d).dtype)
    h = h_bl(fft_size(n, pad), n, lamb, px, d, band_limit)[:, None]
    x = o.astype(np.complex64) if dtype == np.complex64 else o
    return ao.propagate_h(x, h, pad, adjoint, dtype=dtype)


def dudz(o, lamb, d, px, pad=False, band_limit=True, deriv_mask=True):
    """(U, dU/dz), both band-limited: U = crop(ifft2(H mask F)), dU/dz = crop(ifft2(i K kz H mask F)).
    ``deriv_mask=False`` leaves the mask out of the derivative only (a planted defect)."""
    import scipy.fft as sf
    o = np.asarray(o)
    b, _, n, _ = o.shape
    m = fft_size(n, pad)
    p = (m - n) // 2
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    d = np.asarray(d).reshape(-1)
    f = sf.fft2(o.astype(np.complex128)[:, :, idx][:, :, :, idx], workers=-1)
    h = h_bl(m, n, lamb, px, d, band_limit)[:, None]
    hd = h if deriv_mask else h_bl(m, n, lamb, px, d, False)[:, None]
    kz = ao.kz_unshifted(m, n, lamb, px)
    u = sf.ifft2(h * f, workers=-1)[:, :, p:p + n, p:p + n]
    du = sf.ifft2((1j * ao.grad_constant(d) * kz) * hd * f, workers=-1)[:, :, p:p + n, p:p + n]
    return u, du


def z_for_lim(m: int, lamb: float, px: float, lim: int, dtype=np.float64) -> np.ndarray:
    """A distance whose band limit is ``lim``: S / (lamb sqrt(1 + q^2)) = lim + 1/2, half a bin from both neighbours."""
    s = m * px
    r = s / (lamb * (lim + 0.5))
    z = np.asarray(0.5 * s * np.sqrt(max(r * r - 1.0, 0.0)), dtype=dtype)
    got = int(band_limit_mask(m, lamb, px, z)[0][0])
    assert got == lim, (m, lim, got)
    return z


def lim_margin(m: int, lamb: float, px: float, d) -> float:
    """Relative distance of S / (lamb sqrt(1 + q^2)) from the nearest integer: how far a distance is from a jump of lim."""
    z = np.atleast_1d(np.asarray(d)).astype(np.float64)
    s = m * px
    q = 2.0 * z / s
    t = s / (lamb * np.sqrt(1.0 + q * q))
    return float(np.min(np.abs(t - np.round(t)) / t))
