"""Numpy restatement (float64 / complex128) of the reference's angular-spectrum hot path.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Every function cites the reference lines it
follows; paths are relative to the reference checkout (csleemooo/style_transfer_based_holographic_imaging).

The reference evaluates the transfer-function phase as ``(1j*2*pi*d) * G_in`` where ``d`` is an fp32
tensor: the product ``1j*2*pi*d`` is formed first, in complex64, so the phase constant is
``c = fl32(fl32(2*pi) * d)`` and only then promoted to double (utils/Angular_Spectrum_Method.py:29).
``phase_constant`` reproduces exactly that rounding; everything else is carried in double, which is
*more* accurate than the reference (fp32 forward FFT) and agrees with it to ~2e-7 rel-L2.
"""
from __future__ import annotations

import numpy as np

TWO_PI_F32 = np.float32(2.0 * np.pi)


# --------------------------------------------------------------------------------------------
# transfer function
# --------------------------------------------------------------------------------------------
def centred_frequencies(n: int, px: float, zero_padding: bool) -> np.ndarray:
    """Centred (fftshift-order) spatial frequencies of one axis.

    utils/Angular_Spectrum_Method.py:13-14 (padded: ``arange(2n)/2 - n//2``) and :16-17 (plain:
    ``arange(n) - n//2``), both divided by ``n*px`` at :19-20.
    """
    if zero_padding:
        f = np.arange(2 * n, dtype=np.float64) / 2 - n // 2
    else:
        f = np.arange(n, dtype=np.float64) - n // 2
    return f / (n * px)


def kz_centred(n: int, lamb: float, px: float, zero_padding: bool) -> np.ndarray:
    """``sqrt(max(1 - lamb^2 (fx_i^2 + fy_j^2), 0)) / lamb`` on the centred M x M grid.

    utils/Angular_Spectrum_Method.py:22-23.  Row index <-> fx, column index <-> fy; evanescent bins
    are clamped to kz = 0 (so H = 1 there, not 0).
    """
    f = centred_frequencies(n, px, zero_padding)
    g = 1.0 - (lamb ** 2) * (f[:, None] ** 2 + f[None, :] ** 2)
    return np.sqrt((g > 0) * 1 * g) / lamb


def kz_unshifted(m: int, n: int, lamb: float, px: float) -> np.ndarray:
    """Same table on *unshifted* FFT bins: k(u) = u < m/2 ? u : u - m, f = k / (m*px_eff).

    This is the closed form the CUDA kernel follows (SURVEY.md section 8a); for even m it equals
    ``ifftshift(kz_centred)``.  ``m`` is the FFT size (n or 2n).  Padded mode has f = (k/2)/(n*px).
    """
    k = np.arange(m, dtype=np.float64)
    k = np.where(k < m / 2, k, k - m)
    f = (k / 2) / (n * px) if m == 2 * n else k / (n * px)
    g = 1.0 - (lamb ** 2) * (f[:, None] ** 2 + f[None, :] ** 2)
    return np.sqrt(np.maximum(g, 0.0)) / lamb


def phase_constant(d) -> np.ndarray:
    """``c = fl32(fl32(2 pi) * d)`` as float64 for fp32 ``d``; ``2 pi d`` in double for fp64 / python floats.

    utils/Angular_Spectrum_Method.py:29 -- ``1j*2*pi*d`` is a complex64 product when d is an fp32 tensor.
    """
    d = np.asarray(d)
    if d.dtype == np.float32:
        return (TWO_PI_F32 * d).astype(np.float32).astype(np.float64)
    return 2.0 * np.pi * d.astype(np.float64)


def _as_b(d, batch: int) -> np.ndarray:
    d = np.asarray(d)
    if d.ndim == 0:
        d = np.full((batch,), d, dtype=d.dtype if d.dtype in (np.float32, np.float64) else np.float64)
    return d.reshape(batch if d.size == batch else -1)


def replicate_pad(o: np.ndarray, p: int) -> np.ndarray:
    """``F.pad(O, (p,p,p,p), mode='replicate')`` -- utils/Angular_Spectrum_Method.py:12."""
    return np.pad(o, ((0, 0), (0, 0), (p, p), (p, p)), mode="edge")


def replicate_pad_T(x: np.ndarray, n: int, p: int) -> np.ndarray:
    """Adjoint of ``replicate_pad``: fold the borders back onto the edge rows/cols (SURVEY.md 8a row 6)."""
    y = x[:, :, p:p + n, :].copy()
    y[:, :, 0, :] += x[:, :, :p, :].sum(axis=2)
    y[:, :, n - 1, :] += x[:, :, p + n:, :].sum(axis=2)
    z = y[:, :, :, p:p + n].copy()
    z[:, :, :, 0] += y[:, :, :, :p].sum(axis=3)
    z[:, :, :, n - 1] += y[:, :, :, p + n:].sum(axis=3)
    return z


# --------------------------------------------------------------------------------------------
# ASM  (utils/Angular_Spectrum_Method.py:7-36)
# --------------------------------------------------------------------------------------------
def asm(o: np.ndarray, lamb: float, d, px: float, zero_padding: bool = False) -> np.ndarray:
    """Reference op order: pad -> fftshift(fft2) -> * exp(i c kz) -> ifft2(ifftshift) -> centre crop.

    ``o``: [B,C,N,N] complex (or real).  ``d``: fp32 [B,1,1,1] / [B] / scalar (metres).  Returns complex128.
    """
    o = np.asarray(o)
    b, _, sh, sw = o.shape
    if sh != sw:
        raise ValueError("square inputs only (the reference's kz grid does not broadcast otherwise)")
    x = o.astype(np.complex128)
    if zero_padding:
        if sh % 2:
            raise ValueError("odd N with zero_padding is not supported by the reference")
        x = replicate_pad(x, sh // 2)
    kz = kz_centred(sh, lamb, px, zero_padding)                        # :22-23
    c = phase_constant(_as_b(d, b)).reshape(b, 1, 1, 1)                # :29
    h = np.exp(1j * (c * kz[None, None]))                              # :29
    spec = np.fft.fftshift(np.fft.fft2(x), axes=(-2, -1))              # :38-42
    u = np.fft.ifft2(np.fft.ifftshift(h * spec, axes=(-2, -1)))        # :33, :44-48
    m = u.shape[-1]
    lo = (m - sh) // 2                                                  # :50-53
    return u[:, :, lo:lo + sh, lo:lo + sh]


def asm_closed_form(o: np.ndarray, lamb: float, d, px: float, zero_padding: bool = False,
                    conj: bool = False) -> np.ndarray:
    """The kernel's formulation: unshifted bins, replicate pad by index clamp, no fftshift pair.

    ``conj=True`` uses conj(H) (propagation by -z).  Pad handling stays the *forward* one (replicate in,
    crop out); the true adjoint of the padded operator is ``asm_adjoint``.
    """
    o = np.asarray(o)
    b, _, n, _ = o.shape
    m = 2 * n if zero_padding else n
    p = (m - n) // 2
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    x = o.astype(np.complex128)[:, :, idx][:, :, :, idx]
    kz = kz_unshifted(m, n, lamb, px)
    c = phase_constant(_as_b(d, b)).reshape(b, 1, 1, 1)
    theta = c * kz[None, None]
    h = np.exp((-1j if conj else 1j) * theta)
    u = np.fft.ifft2(h * np.fft.fft2(x))
    return u[:, :, p:p + n, p:p + n]


def asm_adjoint(g: np.ndarray, lamb: float, d, px: float, zero_padding: bool = False) -> np.ndarray:
    """Exact adjoint (vector-Jacobian product w.r.t. O, PyTorch convention) of ``asm``.

    grad_O = replicate_pad^T( ifft2( conj(H) * fft2( zero_embed(g) ) ) )   (SURVEY.md 8a row 6).
    Unpadded this is ``asm(g, -d)``.
    """
    g = np.asarray(g).astype(np.complex128)
    b, ch, n, _ = g.shape
    m = 2 * n if zero_padding else n
    p = (m - n) // 2
    ge = np.zeros((b, ch, m, m), dtype=np.complex128)
    ge[:, :, p:p + n, p:p + n] = g
    kz = kz_unshifted(m, n, lamb, px)
    c = phase_constant(_as_b(d, b)).reshape(b, 1, 1, 1)
    h = np.exp(1j * (c * kz[None, None]))
    y = np.fft.ifft2(np.conj(h) * np.fft.fft2(ge))
    return replicate_pad_T(y, n, p) if p else y


def asm_grad_d(o: np.ndarray, g: np.ndarray, lamb: float, d, px: float, zero_padding: bool = False) -> np.ndarray:
    """d<L>/dd for cotangent ``g`` of U = asm(o): Re sum conj(g) * dU/dd, dU/dd = crop ifft2(i 2pi kz H fft2(pad o)).

    The reference gets this from autograd because ``G_in`` stays in the graph
    (utils/Angular_Spectrum_Method.py:28-29); fl32(2 pi) is the constant the reference multiplies d by.
    Returns float64 [B].
    """
    o = np.asarray(o)
    b, _, n, _ = o.shape
    m = 2 * n if zero_padding else n
    p = (m - n) // 2
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    x = o.astype(np.complex128)[:, :, idx][:, :, :, idx]
    kz = kz_unshifted(m, n, lamb, px)
    c = phase_constant(_as_b(d, b)).reshape(b, 1, 1, 1)
    h = np.exp(1j * (c * kz[None, None]))
    du = np.fft.ifft2(1j * kz[None, None] * h * np.fft.fft2(x))[:, :, p:p + n, p:p + n]
    return float(TWO_PI_F32) * np.real(np.conj(np.asarray(g).astype(np.complex128)) * du).sum(axis=(1, 2, 3))


# --------------------------------------------------------------------------------------------
# Holo_Generator / Back_prop  (utils/Forward_model.py)
# --------------------------------------------------------------------------------------------
class Optics:
    """Stand-in for the ``args`` namespace read at utils/Forward_model.py:9-13 and :45-50."""

    def __init__(self, wavelength=532e-9, pixel_size=1.5e-6, phase_normalize=1.0, distance_normalize=1.0,
                 distance_normalize_constant=0.0, amplitude_normalize=1.0, Holo_G_input="amp_pha"):
        self.wavelength = wavelength
        self.pixel_size = pixel_size
        self.phase_normalize = phase_normalize
        self.distance_normalize = distance_normalize
        self.distance_normalize_constant = distance_normalize_constant
        self.amplitude_normalize = amplitude_normalize
        self.Holo_G_input = Holo_G_input


def metres(d, args) -> np.ndarray:
    """``((d + c0) * s) * 1e-3`` in fp32 tensor arithmetic -- utils/Forward_model.py:18 and :53."""
    d = np.asarray(d, dtype=np.float32)
    t = (d + np.float32(args.distance_normalize_constant)).astype(np.float32)
    t = (t * np.float32(args.distance_normalize)).astype(np.float32)
    return (t * np.float32(1e-3)).astype(np.float32)


def object_field(amplitude, phase, args) -> np.ndarray:
    """``amplitude * exp(1j * phase * phase_normalize)`` -- utils/Forward_model.py:20-22 (complex64 there)."""
    ph = (np.asarray(phase, dtype=np.float32) * np.float32(args.phase_normalize)).astype(np.float32)
    return np.asarray(amplitude, dtype=np.float64) * np.exp(1j * ph.astype(np.float64))


def holo_generator(amplitude, phase, d, args, return_field=False, complex_number=False):
    """utils/Forward_model.py:16-39 (``unwrap`` is a CPU skimage post-process and is out of scope)."""
    u = asm(object_field(amplitude, phase, args), args.wavelength, metres(d, args), args.pixel_size,
            zero_padding=True)                                                           # :24
    if return_field:
        return np.abs(u).astype(np.float32), np.angle(u).astype(np.float32)              # :27-34
    if complex_number:
        return u                                                                         # :36-37
    return (np.abs(u) ** 2).astype(np.float32)                                           # :39


def back_prop(holo, d, args) -> np.ndarray:
    """utils/Forward_model.py:52-65.  Returns float64 [B,2,N,N] like the reference."""
    h = np.sqrt(np.asarray(holo, dtype=np.float32))                                      # :55
    u = asm(h, args.wavelength, metres(d, args), args.pixel_size) * args.amplitude_normalize  # :56
    if args.Holo_G_input == "amp_pha":
        r, i = np.abs(u), np.angle(u)                                                    # :58-60
    else:
        r, i = np.real(u), np.imag(u)                                                    # :61-63
    return np.concatenate([r, i], axis=1)                                                # :65


def holo_generator_vjp(amplitude, phase, d, w, args):
    """Gradients of sum(w * Holo_Generator(amplitude, phase, d)) (intensity mode) w.r.t. the three inputs.

    Chain rule of SURVEY.md 8a row 6: g = 2 w U; grad_O = asm_adjoint(g); grad_A = Re(conj(e^{i phi}) grad_O);
    grad_phi = phase_normalize * Im(conj(O) grad_O); grad_d_in = grad_d * distance_normalize * 1e-3.
    Returns (grad_A [B,1,N,N], grad_phi [B,1,N,N], grad_d [B]) in float64.
    """
    o = object_field(amplitude, phase, args)
    z = metres(d, args)
    u = asm(o, args.wavelength, z, args.pixel_size, zero_padding=True)
    g = 2.0 * np.asarray(w, dtype=np.float64) * u
    go = asm_adjoint(g, args.wavelength, z, args.pixel_size, zero_padding=True)
    a = np.asarray(amplitude, dtype=np.float64)
    ph = (np.asarray(phase, dtype=np.float32) * np.float32(args.phase_normalize)).astype(np.float64)
    e = np.exp(1j * ph)
    grad_a = np.real(np.conj(e) * go)
    grad_phi = args.phase_normalize * np.imag(np.conj(o) * go)
    gd = asm_grad_d(o, g, args.wavelength, z, args.pixel_size, zero_padding=True)
    grad_d = gd * float(np.float32(args.distance_normalize)) * float(np.float32(1e-3))
    return grad_a, grad_phi, grad_d


# --------------------------------------------------------------------------------------------
# the C ABI's modes (include/asm_b200.h), the transfer function on its own, and a complex64 pipeline
# --------------------------------------------------------------------------------------------
IN_COMPLEX, IN_AMP_PHASE, IN_SQRT_REAL, IN_COT_FIELD, IN_REAL, IN_CONST_AMP_PHASE = range(6)
OUT_COMPLEX, OUT_INTENSITY, OUT_ABS_ANGLE, OUT_REIM_CAT, OUT_ABSANG_CAT, OUT_GRAD_AP = range(6)


def transfer_function(m: int, n: int, lamb: float, px: float, d) -> np.ndarray:
    """H = exp(i c kz) on the unshifted m x m bins, one table per distance: [len(d), m, m] complex128.

    ``kz_unshifted`` (evanescent bins clamped to kz = 0, so H = 1 there) times ``phase_constant(d)``.
    """
    kz = kz_unshifted(m, n, lamb, px)
    c = phase_constant(np.atleast_1d(d))
    return np.exp(1j * (c[:, None, None] * kz[None]))


def grad_constant(d) -> float:
    """K of dU/dz = ifft2(i K kz H fft2(O)): fl32(2 pi) for fp32 distances, 2 pi for fp64 ones."""
    return float(TWO_PI_F32) if np.asarray(d).dtype == np.float32 else 2.0 * np.pi


def scaled_phase(phase, in_scale) -> np.ndarray:
    """``fl32(phase * in_scale)`` as float64: the phase the library takes sin / cos of."""
    return (np.asarray(phase, dtype=np.float32) * np.float32(in_scale)).astype(np.float32).astype(np.float64)


def input_field(in_mode: int, in0, in1=None, in_scale: float = 1.0) -> np.ndarray:
    """The complex128 field O that ``in_mode`` builds from (in0, in1) (include/asm_b200.h, IN_*)."""
    if in_mode == IN_COMPLEX:
        return np.asarray(in0).astype(np.complex128)
    if in_mode == IN_AMP_PHASE:
        return np.asarray(in0, dtype=np.float64) * np.exp(1j * scaled_phase(in1, in_scale))
    if in_mode == IN_CONST_AMP_PHASE:
        return float(np.asarray(in0).reshape(-1)[0]) * np.exp(1j * scaled_phase(in1, in_scale))
    if in_mode == IN_SQRT_REAL:
        return np.sqrt(np.asarray(in0, dtype=np.float64)).astype(np.complex128)
    if in_mode == IN_COT_FIELD:
        return 2.0 * np.asarray(in0, dtype=np.float64) * np.asarray(in1).astype(np.complex128)
    if in_mode == IN_REAL:
        return np.asarray(in0, dtype=np.float64).astype(np.complex128)
    raise ValueError(f"unknown in_mode {in_mode}")


def _fft_pair(dtype=np.complex128):
    """(fft2, ifft2) over the last two axes: scipy.fft keeps complex128 in double and complex64 in single precision."""
    import scipy.fft as sf
    return (lambda x: sf.fft2(x, workers=-1)), (lambda x: sf.ifft2(x, workers=-1))


def propagate_h(o: np.ndarray, h: np.ndarray, zero_padding: bool = False, adjoint: bool = False,
                dtype=np.complex128) -> np.ndarray:
    """The library's operator with an explicit transfer function ``h`` (broadcast against [B,C,M,M]).

    forward: crop(ifft2(h fft2(replicate_pad(o))));  adjoint: replicate_pad^T(ifft2(conj(h) fft2(zero_embed(o)))).
    ``dtype`` complex64 runs both transforms in single precision with ``h`` rounded to complex64.
    """
    fft2, ifft2 = _fft_pair(dtype)
    o = np.asarray(o)
    b, ch, n, _ = o.shape
    m = 2 * n if zero_padding else n
    p = (m - n) // 2
    h = np.asarray(h).astype(dtype)
    if adjoint:
        x = np.zeros((b, ch, m, m), dtype=dtype)
        x[:, :, p:p + n, p:p + n] = o
        y = ifft2(np.conj(h) * fft2(x)).astype(dtype)
        return replicate_pad_T(y, n, p) if p else y
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    x = o.astype(dtype)[:, :, idx][:, :, :, idx]
    return ifft2(h * fft2(x)).astype(dtype)[:, :, p:p + n, p:p + n]


def _h_per_sample(n: int, zero_padding: bool, lamb: float, d, px: float, batch: int) -> np.ndarray:
    m = 2 * n if zero_padding else n
    return transfer_function(m, n, lamb, px, _as_b(d, batch))[:, None]


def asm_c128(o, lamb, d, px, zero_padding=False, adjoint=False) -> np.ndarray:
    """Forward (``asm_closed_form``) or exact adjoint (``asm_adjoint``) through ``propagate_h`` in float64."""
    o = np.asarray(o)
    h = _h_per_sample(o.shape[-1], zero_padding, lamb, d, px, o.shape[0])
    return propagate_h(o, h, zero_padding, adjoint)


def asm_c64(o, lamb, d, px, zero_padding=False, adjoint=False) -> np.ndarray:
    """The same operator as a plain complex64 pipeline: single-precision FFTs, H rounded to complex64.

    A correct single-precision implementation; its distance from the float64 result calibrates the bounds of the
    GPU parity tests (about 2-4e-7 rel-L2 on white fields).
    """
    o = np.asarray(o)
    h = _h_per_sample(o.shape[-1], zero_padding, lamb, d, px, o.shape[0])
    return propagate_h(o.astype(np.complex64), h, zero_padding, adjoint, dtype=np.complex64)


def output_stage(u: np.ndarray, out_mode: int, out_scale: float = 1.0) -> list:
    """What asm_b200_forward writes for ``out_mode`` (out0, then out1), computed in the precision of ``u``."""
    real = np.float32 if u.dtype == np.complex64 else np.float64
    s = real(out_scale)
    if out_mode == OUT_COMPLEX:
        return [u]
    if out_mode == OUT_INTENSITY:
        return [np.abs(u) ** 2, u]
    if out_mode == OUT_ABS_ANGLE:
        return [np.abs(u), np.angle(u)]
    if out_mode == OUT_REIM_CAT:
        return [np.concatenate([u.real * s, u.imag * s], axis=1)]
    if out_mode == OUT_ABSANG_CAT:
        su = u * s
        return [np.concatenate([np.abs(su), np.angle(su)], axis=1)]
    raise ValueError(f"out_mode {out_mode} is not a forward output")


def grad_ap(go: np.ndarray, amplitude, phase, in_scale: float) -> list:
    """OUT_GRAD_AP of the adjoint: [Re(conj(e) go), in_scale a Im(conj(e) go)], e = exp(i fl32(phase in_scale))."""
    e = np.exp(1j * scaled_phase(phase, in_scale)).astype(go.dtype)
    t = np.conj(e) * go
    real = t.real.dtype.type
    return [t.real, real(in_scale) * np.asarray(amplitude).astype(real) * t.imag]


def asm_dudz(o, lamb, d, px, zero_padding=False):
    """(U, dU/dz) from one spectrum: U = crop(ifft2(H F)), dU/dz = crop(ifft2(i K kz H F)), F = fft2(pad(o)), K =
    ``grad_constant(d)``.  complex128 [B,C,N,N] each."""
    o = np.asarray(o)
    b, _, n, _ = o.shape
    m = 2 * n if zero_padding else n
    p = (m - n) // 2
    idx = np.clip(np.arange(m) - p, 0, n - 1)
    fft2, ifft2 = _fft_pair()
    d = _as_b(d, b)
    hf = transfer_function(m, n, lamb, px, d)[:, None] * fft2(o.astype(np.complex128)[:, :, idx][:, :, :, idx])
    u = ifft2(hf)[:, :, p:p + n, p:p + n]
    du = ifft2((1j * grad_constant(d) * kz_unshifted(m, n, lamb, px)) * hf)[:, :, p:p + n, p:p + n]
    return u, du


def grad_z_sum(g, u, du, lamb, d, kshift=0.0):
    """grad_z[b] = Re sum_{c,y,x} conj(g) dU/dz and its rounding scale S_b = sum |Re(conj(g) dU/dz)|, float64 [B] each.

    With kshift = 1 the derivative is taken with kz - 1/lamb in place of kz, i.e. dU/dz - i K U / lamb: the form the
    library evaluates for the intensity cotangent (asm_b200_grad_z).  It gives the same gradient when g = 2 w U.
    """
    if kshift:
        du = du - (1j * grad_constant(d) * kshift / lamb) * u
    t = np.real(np.conj(np.asarray(g).astype(np.complex128)) * du)
    return t.sum(axis=(1, 2, 3)), np.abs(t).sum(axis=(1, 2, 3))


def asm_grad_z(o, g, lamb, d, px, zero_padding=False, kshift=0.0):
    """``grad_z_sum`` of U = asm(o) (see there): returns (grad [B], S [B])."""
    u, du = asm_dudz(o, lamb, d, px, zero_padding)
    return grad_z_sum(g, u, du, lamb, np.asarray(_as_b(d, np.asarray(o).shape[0])), kshift)


def rel_l2(a, b) -> float:
    a = np.asarray(a)
    b = np.asarray(b)
    den = np.linalg.norm(b.ravel())
    return float(np.linalg.norm((a - b).ravel()) / (den if den > 0 else 1.0))
