"""Focal stacks, focus metrics and autofocus over the C ABI's ``asm_b200_focal_stack``.

One hologram propagated to many distances: the forward row FFT of every sample runs once and is shared by all of its
planes, and the moments (Sum |U|, Sum |U|^2, Sum |U|^4 per plane) are reduced on the device, so an autofocus sweep
never materialises the [B, K, N, N] stack.  Plane (b, k) equals ``ASM(x[b], z[b, k])`` (``asm_forward_raw``).

No autograd: ``ASM`` is the differentiable path.  CUDA tensors only, as everywhere in this package.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple, Union

import torch

from . import _lib as L
from .functional import _c64, _f32, _ptr, _stream

_OUT_MODES = {"intensity": L.OUT_INTENSITY, "complex": L.OUT_COMPLEX, "abs_angle": L.OUT_ABS_ANGLE, None: None}


def _stack_distances(z, b: int, device: torch.device) -> Tuple[torch.Tensor, int, int]:
    """[K] (shared by all samples) or [B, K] distances in metres -> contiguous [B, K] tensor, z_dtype, K.
    fp32 tensors keep the reference's complex64 phase constant; fp64 tensors and python sequences use the double one
    (as ``functional.prepare_distance``)."""
    if isinstance(z, torch.Tensor):
        zt = z.detach()
        zd = L.Z_F64 if zt.dtype == torch.float64 else L.Z_F32
        zt = zt.to(device=device, dtype=torch.float64 if zd == L.Z_F64 else torch.float32)
    else:
        zt, zd = torch.tensor([float(v) for v in z], dtype=torch.float64, device=device), L.Z_F64
    if zt.dim() == 1 and zt.numel() > 0:
        zt = zt.reshape(1, -1).expand(b, -1)
    elif not (zt.dim() == 2 and zt.shape[0] == b and zt.shape[1] > 0):
        raise RuntimeError(f"z must be [K] or [B, K] with B = {b}; got shape {tuple(zt.shape)}")
    return zt.contiguous(), zd, int(zt.shape[1])


def focal_stack(x: torch.Tensor, z: Union[torch.Tensor, Sequence[float]], wavelength: float, pixel_size: float,
                zero_padding: bool = False, *, hologram: bool = False, output: Optional[str] = "intensity",
                moments: bool = False):
    """Propagate every sample of ``x`` to K distances.

    x: [B, 1, N, N] or [B, N, N]; complex64 field, real field, or (``hologram=True``) an intensity whose square root is
       the field (as ``Back_prop``).
    z: [K] or [B, K] distances in metres.
    output: "intensity" (fp32 [B, K, N, N]), "complex" (complex64), "abs_angle" (tuple of fp32 |U|, angle(U)) or None.
    moments: also return the float64 [B, K, 3] moments (Sum |U|, Sum |U|^2, Sum |U|^4) over each N x N plane.
    Returns the images, ``(images, moments)``, or only the moments when ``output`` is None.
    """
    if output not in _OUT_MODES:
        raise ValueError(f"output must be one of 'intensity', 'complex', 'abs_angle' or None; got {output!r}")
    if output is None and not moments:
        raise ValueError("output=None needs moments=True: there would be nothing to return")
    if not isinstance(x, torch.Tensor):
        raise TypeError("x must be a torch.Tensor")
    if torch.is_grad_enabled() and (x.requires_grad or (isinstance(z, torch.Tensor) and z.requires_grad)):
        raise RuntimeError("focal_stack is not differentiable; use ASM for gradients through the propagation")
    if not x.is_cuda:
        raise RuntimeError(f"x is on {x.device}: the B200 ASM propagator has no CPU fallback (move it to a CUDA device)")
    if x.dim() == 4:
        if x.shape[1] != 1:
            raise RuntimeError(f"x must be [B, 1, N, N] or [B, N, N]; got shape {tuple(x.shape)}")
        x = x[:, 0]
    if x.dim() != 3 or x.shape[1] != x.shape[2]:
        raise RuntimeError(f"x must be [B, 1, N, N] or [B, N, N] with square planes; got shape {tuple(x.shape)}")
    b, n = int(x.shape[0]), int(x.shape[1])
    if hologram:
        if x.is_complex():
            raise RuntimeError("hologram=True takes a real intensity")
        xin, in_mode = _f32(x), L.IN_SQRT_REAL
    elif x.is_complex():
        xin, in_mode = _c64(x), L.IN_COMPLEX
    else:
        xin, in_mode = _f32(x), L.IN_REAL
    dev = xin.device
    zt, zd, k = _stack_distances(z, b, dev)
    lib = L.load()
    with torch.cuda.device(dev):
        nbytes = lib.asm_b200_focal_stack_workspace_bytes(b, k, n, int(zero_padding))
    if nbytes == 0:
        raise RuntimeError(f"unsupported focal stack: B={b}, K={k}, N={n}, zero_padding={zero_padding}")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out_mode = _OUT_MODES[output]
    out0 = out1 = None
    if output == "complex":
        out0 = torch.empty((b, k, n, n), dtype=torch.complex64, device=dev)
    elif output is not None:
        out0 = torch.empty((b, k, n, n), dtype=torch.float32, device=dev)
        if output == "abs_angle":
            out1 = torch.empty((b, k, n, n), dtype=torch.float32, device=dev)
    mom = torch.empty((b, k, 3), dtype=torch.float64, device=dev) if moments else None
    with torch.cuda.device(dev):
        rc = lib.asm_b200_focal_stack(_ptr(xin), None, _ptr(zt), zd, k, _ptr(out0), _ptr(out1), _ptr(mom), b, n,
                                      int(zero_padding), in_mode, L.OUT_INTENSITY if out_mode is None else out_mode,
                                      float(wavelength), float(pixel_size), 1.0, _ptr(ws), ws.numel(), _stream())
    L.check(rc)
    images = (out0, out1) if output == "abs_angle" else out0
    if output is None:
        return mom
    return (images, mom) if moments else images


def focus_metric(moments: torch.Tensor, n_pixels: int, metric: str = "tamura") -> torch.Tensor:
    """Sharpness of each plane from its moments [..., 3] (float64).

    "tamura":   sqrt(std / mean) of the amplitude |U| (Tamura coefficient; Memmolo et al., Opt. Lett. 36, 2011).
    "variance": normalised variance of the intensity, (<I^2> - <I>^2) / <I>^2.
    """
    m = moments.to(torch.float64) / float(n_pixels)
    if metric == "tamura":
        mean = m[..., 0]
        std = torch.sqrt(torch.clamp(m[..., 1] - mean * mean, min=0.0))
        return torch.sqrt(std / mean)
    if metric == "variance":
        return (m[..., 2] - m[..., 1] * m[..., 1]) / (m[..., 1] * m[..., 1])
    raise ValueError(f"metric must be 'tamura' or 'variance'; got {metric!r}")


def autofocus(x: torch.Tensor, z: Union[torch.Tensor, Sequence[float]], wavelength: float, pixel_size: float,
              zero_padding: bool = False, *, hologram: bool = True, metric: str = "tamura", select: str = "min"):
    """Pick, per sample, the candidate distance whose plane is extreme in ``metric``.

    One moments-only focal stack: no [B, K, N, N] tensor is allocated.  ``select`` is "min" or "max": a pure-phase
    object has its most uniform amplitude at focus, so its Tamura coefficient (or normalised variance) is smallest
    there ("min"); absorbing objects are usually sharpest at the maximum ("max").
    Returns (z_best [B] in the dtype of the distances, index [B] int64, curve [B, K] float64).
    """
    if select not in ("min", "max"):
        raise ValueError(f"select must be 'min' or 'max'; got {select!r}")
    mom = focal_stack(x, z, wavelength, pixel_size, zero_padding, hologram=hologram, output=None, moments=True)
    n = x.shape[-1]
    curve = focus_metric(mom, n * n, metric)
    index = torch.argmin(curve, dim=1) if select == "min" else torch.argmax(curve, dim=1)
    zt, _, _ = _stack_distances(z, mom.shape[0], mom.device)
    z_best = torch.gather(zt, 1, index.reshape(-1, 1)).reshape(-1)
    return z_best, index, curve
