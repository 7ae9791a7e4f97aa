"""Drop-in for the reference's ``utils/Angular_Spectrum_Method.py`` on B200.

Same call signature as the reference's ``ASM`` (``utils/Angular_Spectrum_Method.py:7``); the padded /
unpadded propagation runs in the fused sm_100a pipeline instead of ~12 torch launches.

Documented deviations (SURVEY.md section 8b):
  * CUDA tensors only -- there is no CPU fallback; CPU tensors raise ``RuntimeError``.
  * the result is complex64 (the reference's complex128 is an accident of its float64 numpy grid);
    pass ``ref_dtype=True`` to upcast.
  * only square power-of-two fields with 32 <= FFT size <= 4096 (the reference itself rejects non-square).
  * ``band_limit=True`` (opt-in, not in the reference) applies the band-limited angular spectrum of Matsushima &
    Shimobaba (Opt. Express 17, 19662, 2009): bins with |f_x| or |f_y| > 1 / (lamb sqrt(1 + (2 d / (M px))^2)) get
    H = 0, M the FFT size.  It removes the aliasing of the undersampled chirp at long distances; at short ones (where
    the limit keeps every bin) the result is bit-identical to the plain call.  The distance gradient treats the mask as
    constant: the loss jumps where the limit changes, and the gradient does not see those jumps.
  * ``requires_grad`` is accepted for signature compatibility; gradients flow to ``O`` and ``d`` whenever they
    require grad, exactly like the reference's autograd graph, but the output does not spuriously require
    grad for non-differentiable inputs.
"""
from __future__ import annotations

import torch

from .functional import AsmPropagate


def ASM(O, lamb, d, px, requires_grad=True, zero_padding=False, ref_dtype=False, band_limit=False):
    U = AsmPropagate.apply(O, d, float(lamb), float(px), bool(zero_padding), bool(band_limit))
    return U.to(torch.complex128) if ref_dtype else U


def torch_fft(H):
    """``fftshift(fft2(H))`` -- utils/Angular_Spectrum_Method.py:38-42 (helper, not on the fused path)."""
    return torch.fft.fftshift(torch.fft.fft2(H), dim=(-2, -1))


def torch_ifft(H):
    """``ifft2(ifftshift(H))`` -- utils/Angular_Spectrum_Method.py:44-48 (helper, not on the fused path)."""
    return torch.fft.ifft2(torch.fft.ifftshift(H, dim=(-2, -1)))


def center_crop(H, size):
    """Centre crop of the last two dims -- utils/Angular_Spectrum_Method.py:50-53."""
    nh, nw = H.shape[-2], H.shape[-1]
    return H[:, :, (nh - size) // 2:(nh + size) // 2, (nw - size) // 2:(nw + size) // 2]
