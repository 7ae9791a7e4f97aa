"""Drop-in for the reference's ``utils/Forward_model.py`` on B200: ``Holo_Generator`` and ``Back_prop``.

Constructor and ``forward`` signatures are those of the reference (``utils/Forward_model.py:6-16`` and
``:42-52``); ``args`` is any object with the same attributes.  Both modules have no parameters, so
``.to(device)`` stays a no-op (``test_field_retrieval_mnist.py:94``).

Deviations (SURVEY.md section 8b): CUDA tensors only; ``complex_number=True`` returns complex64 and
``Back_prop`` returns float32 (reference: complex128 / float64) unless ``ref_dtype=True`` is set on the module.
``band_limit=True`` on either constructor (opt-in, not in the reference) propagates with the band-limited angular
spectrum (see ``ASM``); the ``forward`` signatures stay the reference's.
"""
from __future__ import annotations

import torch
from torch import nn

from . import functional as F_
from .Angular_Spectrum_Method import ASM, center_crop  # noqa: F401  (re-exported like the reference module)


def unwrap(x: torch.Tensor) -> torch.Tensor:
    """2-D phase unwrapping of every image of ``x`` ([B, 1, H, W] or [B, H, W]) on the device, stream-ordered: the
    replacement of ``utils/functions.py:44-59`` (a ``.cpu()`` sync and one ``skimage.restoration.unwrap_phase`` call per
    image).  Same algorithm (Herraez et al. 2002, reliability-sorted edges); returns [B, 1, H, W] float32 on ``x.device``
    (the reference returns a float64 CPU tensor: its callers move it back with ``.to(device).float()``)."""
    return F_.unwrap_phase(x)


def _broadcast_amp_phase(amplitude, phase):
    """``amplitude*torch.exp(1j*phase)`` (utils/Forward_model.py:22) broadcasts its operands; so do we, through
    ``torch.broadcast_tensors`` so that autograd sum-reduces the gradients of broadcast inputs itself.  A one-element
    amplitude (python scalar, 0-dim or [1,1,1,1] tensor) stays a scalar: the kernels take it as a constant."""
    if not isinstance(phase, torch.Tensor):
        raise TypeError("phase must be a torch.Tensor")
    if not isinstance(amplitude, torch.Tensor):
        amplitude = torch.tensor(float(amplitude), dtype=torch.float32, device=phase.device)
    if amplitude.numel() == 1:
        if phase.dim() < 4:
            phase = phase.reshape((1,) * (4 - phase.dim()) + tuple(phase.shape))
        return amplitude, phase
    amplitude, phase = torch.broadcast_tensors(amplitude, phase)
    return amplitude, phase


class Holo_Generator(nn.Module):
    """Free-space forward model: complex object field -> hologram at distance d (utils/Forward_model.py:6-39)."""

    def __init__(self, args, ref_dtype: bool = False, band_limit: bool = False):
        super().__init__()
        self.wavelength = args.wavelength
        self.pixel_size = args.pixel_size
        self.distance_normalize = args.distance_normalize
        self.distance_normalize_constant = args.distance_normalize_constant
        self.phase_normalize = args.phase_normalize
        self.ref_dtype = ref_dtype
        self.band_limit = bool(band_limit)

    def forward(self, amplitude, phase, d, return_field=False, complex_number=False, unwrap=False):
        # normalised mm -> metres with the reference's fp32 rounding sequence (utils/Forward_model.py:18)
        d = ((d + self.distance_normalize_constant) * self.distance_normalize) * 1e-3
        lamb, px, pn, bl = self.wavelength, self.pixel_size, self.phase_normalize, self.band_limit
        amplitude, phase = _broadcast_amp_phase(amplitude, phase)
        needs_graph = torch.is_grad_enabled() and any(
            isinstance(t, torch.Tensor) and t.requires_grad for t in (amplitude, phase, d))
        if return_field:
            if needs_graph:
                U = F_.HoloField.apply(amplitude, phase, d, lamb, px, pn, True, bl)
                amp_prop, ph_prop = torch.abs(U), torch.angle(U)
            else:
                amp_prop, ph_prop = F_.holo_abs_angle(amplitude, phase, d, lamb, px, pn, True, bl)
            if unwrap:
                ph_prop = F_.unwrap_phase(ph_prop)        # (the keyword argument shadows the module-level unwrap)
            return amp_prop, ph_prop
        if complex_number:
            U = F_.HoloField.apply(amplitude, phase, d, lamb, px, pn, True, bl)
            return U.to(torch.complex128) if self.ref_dtype else U
        return F_.HoloIntensity.apply(amplitude, phase, d, lamb, px, pn, True, bl)

    @torch.no_grad()
    def forward_pair(self, amplitude, phase_a, phase_b, d_a, d_b):
        """The hologram-synthesis pattern of ``utils/Data_loader.py:31-32`` / ``:61-67`` (SURVEY.md section 8f row 2):
        two no-grad intensity calls sharing one amplitude, ``model_forward(amplitude, phase_style, d_style)`` and
        ``model_forward(amplitude, phase_content, d_content)``.  Nothing is concatenated: each phase tensor is read in
        place, a constant amplitude (Data_loader.py:25 builds ``torch.ones_like(...)*0.6``; pass ``0.6`` or a one-element
        tensor instead) travels as ONE device scalar (``IN_CONST_AMP_PHASE``: no amplitude plane is read), and both
        results land in one allocation.
        Returns ``(holo_a, holo_b)`` as detached fp32 tensors, exactly what ``.float().detach()`` leaves there."""
        d_a = ((d_a + self.distance_normalize_constant) * self.distance_normalize) * 1e-3
        d_b = ((d_b + self.distance_normalize_constant) * self.distance_normalize) * 1e-3
        amp_a, phase_a = _broadcast_amp_phase(amplitude, phase_a)
        amp_b, phase_b = _broadcast_amp_phase(amplitude, phase_b)
        if amp_a.numel() == 1 or amp_a.data_ptr() == amp_b.data_ptr():
            return F_.holo_intensity_pair(amp_a, phase_a, phase_b, d_a, d_b, self.wavelength, self.pixel_size,
                                          self.phase_normalize, True, self.band_limit)
        return (F_.HoloIntensity.apply(amp_a, phase_a, d_a, self.wavelength, self.pixel_size, self.phase_normalize, True,
                                       self.band_limit),
                F_.HoloIntensity.apply(amp_b, phase_b, d_b, self.wavelength, self.pixel_size, self.phase_normalize, True,
                                       self.band_limit))


class Back_prop(nn.Module):
    """Back-propagated hologram as network input (utils/Forward_model.py:42-65)."""

    def __init__(self, args, ref_dtype: bool = False, band_limit: bool = False):
        super().__init__()
        self.amplitude_normalize = args.amplitude_normalize
        self.wavelength = args.wavelength
        self.pixel_size = args.pixel_size
        self.distance_normalize = args.distance_normalize
        self.distance_normalize_constant = args.distance_normalize_constant
        self.input_type = args.Holo_G_input
        self.ref_dtype = ref_dtype
        self.band_limit = bool(band_limit)

    def forward(self, holo, d):
        d = ((d + self.distance_normalize_constant) * self.distance_normalize) * 0.001
        amp_pha = self.input_type == 'amp_pha'
        needs_graph = torch.is_grad_enabled() and any(
            isinstance(t, torch.Tensor) and t.requires_grad for t in (holo, d))
        if needs_graph:
            U = ASM(torch.sqrt(holo), self.wavelength, d, self.pixel_size, band_limit=self.band_limit) * self.amplitude_normalize
            r, i = (torch.abs(U), torch.angle(U)) if amp_pha else (torch.real(U), torch.imag(U))
            out = torch.cat([r, i], dim=1)
        else:
            out = F_.back_prop_fused(holo, d, self.wavelength, self.pixel_size, self.amplitude_normalize, amp_pha,
                                     self.band_limit)
        return out.to(torch.float64) if self.ref_dtype else out
