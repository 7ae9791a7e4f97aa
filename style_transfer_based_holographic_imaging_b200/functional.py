"""torch.autograd.Functions over the C ABI (include/asm_b200.h).

Everything here is plumbing: tensors are validated, made contiguous, and their device pointers handed to
``libasm_b200.so`` on the current CUDA stream.  There is NO CPU fallback -- CPU tensors raise.

Reference semantics (paths relative to the reference checkout):
  * ``utils/Angular_Spectrum_Method.py:7-36``  ASM
  * ``utils/Forward_model.py:16-39``            Holo_Generator.forward
  * ``utils/Forward_model.py:52-65``            Back_prop.forward
  * the backward PyTorch autograd derives from those (SURVEY.md section 8a row 6).
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib as L


# ---------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------
def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check_field(x: torch.Tensor, name: str) -> Tuple[int, int, int]:
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not x.is_cuda:
        raise RuntimeError(f"{name} is on {x.device}: the B200 ASM propagator has no CPU fallback (move it to a CUDA device)")
    if x.dim() != 4:
        raise RuntimeError(f"{name} must be [B, C, N, N], got shape {tuple(x.shape)}")
    b, c, h, w = x.shape
    if h != w:
        raise RuntimeError(f"{name}: only square fields are supported (got {h}x{w}), as in the reference's kz grid")
    return b, c, h


def prepare_distance(d, batch: int, device: torch.device) -> Tuple[torch.Tensor, int]:
    """Distance in metres -> contiguous [B] tensor + z_dtype.  fp32 tensors keep the reference's complex64
    phase constant; python floats / fp64 tensors use the double one (utils/Angular_Spectrum_Method.py:29)."""
    if isinstance(d, torch.Tensor):
        if d.dtype == torch.float64:
            z, zd = d, L.Z_F64
        else:
            z, zd = d.to(torch.float32), L.Z_F32
        if z.device != device:
            z = z.to(device)
        if z.numel() == 1:
            z = z.reshape(1).expand(batch)
        elif z.numel() == batch and (z.dim() == 1 or tuple(z.shape[1:]) == (1,) * (z.dim() - 1)):
            z = z.reshape(batch)
        else:
            raise RuntimeError(f"distance must be a scalar or [B,1,1,1]; got shape {tuple(d.shape)} for batch {batch}")
        return z.contiguous(), zd
    z = torch.full((batch,), float(d), dtype=torch.float64, device=device)
    return z, L.Z_F64


def _workspace(b: int, c: int, n: int, pad: bool, device: torch.device) -> torch.Tensor:
    with torch.cuda.device(device):     # the size depends on the SM count of the device the call will run on
        nbytes = L.load().asm_b200_workspace_bytes(b, c, n, int(pad))
    if nbytes == 0:
        raise RuntimeError(
            f"unsupported field size N={n} (zero_padding={pad}): N must be a power of two with 32 <= FFT size <= 4096, "
            f"or any other even N with FFT size <= 2048")
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


# band_limit=True: the band-limited transfer function of include/asm_b200.h (asm_b200_*_bl): bins outside
# |f_x|, |f_y| <= 1 / (lambda sqrt(1 + (2 z / (M px))^2)) get H = 0 (Matsushima & Shimobaba 2009).  Opt-in everywhere;
# without it the plain entry point is called, exactly as before the option existed.
def _entry(name: str, band_limit: bool):
    """(C function, trailing arguments): the plain entry point, or its _bl variant with band_limit = 1."""
    lib = L.load()
    if not band_limit:
        return getattr(lib, name), ()
    if not hasattr(lib, name + "_bl"):
        raise L.AsmB200Error(f"{L.LIB_PATH} has no {name}_bl: rebuild it (band_limit=True needs the band-limited entry points)")
    return getattr(lib, name + "_bl"), (1,)


def _forward_call(in0, in1, z, zd, out0, out1, b, c, n, pad, in_mode, out_mode, lamb, px, in_scale, out_scale,
                  band_limit=False):
    ws = _workspace(b, c, n, pad, in0.device)
    with torch.cuda.device(in0.device):
        fn, bl = _entry("asm_b200_forward", band_limit)
        rc = fn(_ptr(in0), _ptr(in1), _ptr(z), zd, _ptr(out0), _ptr(out1), b, c, n, int(pad), in_mode, out_mode,
                float(lamb), float(px), float(in_scale), float(out_scale), _ptr(ws), ws.numel(), _stream(), *bl)
    L.check(rc)


def _adjoint_call(in0, in1, z, zd, aux0, aux1, out0, out1, b, c, n, pad, in_mode, out_mode, lamb, px, in_scale,
                  band_limit=False):
    ws = _workspace(b, c, n, pad, in0.device)
    with torch.cuda.device(in0.device):
        fn, bl = _entry("asm_b200_adjoint", band_limit)
        rc = fn(_ptr(in0), _ptr(in1), _ptr(z), zd, _ptr(aux0), _ptr(aux1), _ptr(out0), _ptr(out1), b, c, n, int(pad),
                in_mode, out_mode, float(lamb), float(px), float(in_scale), _ptr(ws), ws.numel(), _stream(), *bl)
    L.check(rc)


def _grad_z_call(in0, in1, z, zd, cot0, cot1, cot_mode, b, c, n, pad, in_mode, lamb, px, in_scale,
                 band_limit=False) -> torch.Tensor:
    ws = _workspace(b, c, n, pad, in0.device)
    gz = torch.empty(b, dtype=torch.float64, device=in0.device)
    with torch.cuda.device(in0.device):
        fn, bl = _entry("asm_b200_grad_z", band_limit)
        rc = fn(_ptr(in0), _ptr(in1), _ptr(z), zd, _ptr(cot0), _ptr(cot1), cot_mode, _ptr(gz), b, c, n, int(pad),
                in_mode, float(lamb), float(px), float(in_scale), _ptr(ws), ws.numel(), _stream(), *bl)
    L.check(rc)
    return gz


def _amp_phase(amplitude, phase):
    """(amplitude f32, phase f32, in_mode): a one-element amplitude (the loaders' constant 0.6, utils/Data_loader.py:25)
    is passed as a device scalar and never expanded (IN_CONST_AMP_PHASE: 4 B/pixel less HBM traffic); otherwise both
    planes are full [B,C,N,N] fields (Holo_Generator.forward has already broadcast them like the reference's
    ``amplitude*torch.exp(1j*phase)``)."""
    if amplitude.device != phase.device:
        raise RuntimeError("amplitude and phase must be on the same CUDA device")
    ph = _f32(phase)
    if amplitude.numel() == 1:
        return _f32(amplitude).reshape(1), ph, L.IN_CONST_AMP_PHASE
    if tuple(amplitude.shape) != tuple(phase.shape):
        raise RuntimeError(f"amplitude {tuple(amplitude.shape)} and phase {tuple(phase.shape)} must be broadcast first")
    return _f32(amplitude), ph, L.IN_AMP_PHASE


def _c64(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.complex64).contiguous()


def _f32(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).contiguous()


def _z_meta(z):
    """(shape, dtype) of a tensor distance argument -- all the backward needs to shape its gradient; None for floats."""
    return (tuple(z.shape), z.dtype) if isinstance(z, torch.Tensor) else None


def _grad_like(g: torch.Tensor, z_meta) -> Optional[torch.Tensor]:
    """grad for the distance argument in the shape/dtype it came in."""
    if z_meta is None:
        return None
    shape, dtype = z_meta
    numel = 1
    for d in shape:
        numel *= d
    if numel == 1 and g.numel() != 1:
        g = g.sum()
    return g.to(dtype).reshape(shape)


# ---------------------------------------------------------------------------------------------------
# raw (non-differentiable) entry points -- also what bench.py times
# ---------------------------------------------------------------------------------------------------
def asm_forward_raw(field: torch.Tensor, z, lamb: float, px: float, pad: bool, out_mode: int = L.OUT_COMPLEX,
                    out: Optional[torch.Tensor] = None, band_limit: bool = False) -> torch.Tensor:
    """complex64 (or real fp32) [B,C,N,N] -> complex64 field or fp32 intensity, one fused pipeline."""
    b, c, n = _check_field(field, "O")
    if field.is_complex():
        x, in_mode = _c64(field), L.IN_COMPLEX
    else:
        x, in_mode = _f32(field), L.IN_REAL
    zt, zd = prepare_distance(z, b, x.device)
    if out is None:
        out = torch.empty((b, c, n, n), device=x.device,
                          dtype=torch.complex64 if out_mode == L.OUT_COMPLEX else torch.float32)
    _forward_call(x, None, zt, zd, out, None, b, c, n, pad, in_mode, out_mode, lamb, px, 1.0, 1.0, band_limit)
    return out


def asm_adjoint_raw(g: torch.Tensor, z, lamb: float, px: float, pad: bool, out: Optional[torch.Tensor] = None,
                    band_limit: bool = False) -> torch.Tensor:
    """Adjoint propagation of a complex64 cotangent (exact VJP of ASM w.r.t. O)."""
    b, c, n = _check_field(g, "cotangent")
    x = _c64(g)
    zt, zd = prepare_distance(z, b, x.device)
    if out is None:
        out = torch.empty_like(x)
    _adjoint_call(x, None, zt, zd, None, None, out, None, b, c, n, pad, L.IN_COMPLEX, L.OUT_COMPLEX, lamb, px, 1.0,
                  band_limit)
    return out


# ---------------------------------------------------------------------------------------------------
# autograd
# ---------------------------------------------------------------------------------------------------
class AsmPropagate(torch.autograd.Function):
    """U = ASM(O, lamb, z, px, zero_padding)  -- complex64 out (the reference returns complex128)."""

    @staticmethod
    def forward(ctx, field, z, lamb, px, pad, band_limit=False):
        b, c, n = _check_field(field, "O")
        if field.is_complex():
            x, in_mode = _c64(field), L.IN_COMPLEX
        else:
            x, in_mode = _f32(field), L.IN_REAL
        zt, zd = prepare_distance(z, b, x.device)
        out = torch.empty((b, c, n, n), dtype=torch.complex64, device=x.device)
        _forward_call(x, None, zt, zd, out, None, b, c, n, pad, in_mode, L.OUT_COMPLEX, lamb, px, 1.0, 1.0, band_limit)
        z_meta = _z_meta(z)
        need_z = z_meta is not None and ctx.needs_input_grad[1]
        ctx.save_for_backward(x if need_z else None, zt)      # the field is only needed for the distance gradient
        ctx.meta = (b, c, n, bool(pad), float(lamb), float(px), zd, in_mode, field.dtype, z_meta, bool(band_limit))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        x, zt = ctx.saved_tensors
        b, c, n, pad, lamb, px, zd, in_mode, in_dtype, z_meta, bl = ctx.meta
        g = _c64(grad_out)
        grad_field = grad_z = None
        if ctx.needs_input_grad[0]:
            go = torch.empty_like(g)
            _adjoint_call(g, None, zt, zd, None, None, go, None, b, c, n, pad, L.IN_COMPLEX, L.OUT_COMPLEX, lamb, px, 1.0,
                          bl)
            grad_field = go.to(in_dtype) if in_dtype.is_complex else go.real.to(in_dtype)
        if ctx.needs_input_grad[1] and z_meta is not None and x is not None:
            gz = _grad_z_call(x, None, zt, zd, g, None, L.IN_COMPLEX, b, c, n, pad, in_mode, lamb, px, 1.0, bl)
            grad_z = _grad_like(gz, z_meta)
        return grad_field, grad_z, None, None, None, None


class HoloField(torch.autograd.Function):
    """U = ASM(A exp(i phase pn), z, zero_padding=True) as complex64 (utils/Forward_model.py:20-24)."""

    @staticmethod
    def forward(ctx, amplitude, phase, z, lamb, px, phase_normalize, pad, band_limit=False):
        b, c, n = _check_field(phase, "phase")
        a, ph, in_mode = _amp_phase(amplitude, phase)
        zt, zd = prepare_distance(z, b, ph.device)
        out = torch.empty((b, c, n, n), dtype=torch.complex64, device=ph.device)
        _forward_call(a, ph, zt, zd, out, None, b, c, n, pad, in_mode, L.OUT_COMPLEX, lamb, px, phase_normalize, 1.0,
                      band_limit)
        ctx.save_for_backward(a, ph, zt)
        ctx.meta = (b, c, n, bool(pad), float(lamb), float(px), zd, float(phase_normalize), amplitude.dtype, phase.dtype,
                    _z_meta(z), in_mode, tuple(amplitude.shape), bool(band_limit))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        a, ph, zt = ctx.saved_tensors
        b, c, n, pad, lamb, px, zd, pn, adt, pdt, z_meta, in_mode, ashape, bl = ctx.meta
        g = _c64(grad_out)
        ga = gp = gz = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            af = a if in_mode == L.IN_AMP_PHASE else a.expand(ph.shape).contiguous()
            ga = torch.empty_like(af)
            gp = torch.empty_like(ph)
            _adjoint_call(g, None, zt, zd, af, ph, ga, gp, b, c, n, pad, L.IN_COMPLEX, L.OUT_GRAD_AP, lamb, px, pn, bl)
            ga = (ga if in_mode == L.IN_AMP_PHASE else ga.sum().reshape(ashape)).to(adt)
            gp = gp.to(pdt)
        if ctx.needs_input_grad[2] and z_meta is not None:
            gz = _grad_like(_grad_z_call(a, ph, zt, zd, g, None, L.IN_COMPLEX, b, c, n, pad, in_mode, lamb, px, pn, bl),
                            z_meta)
        return ga, gp, gz, None, None, None, None, None


class HoloIntensity(torch.autograd.Function):
    """I = |ASM(A exp(i phase pn), z, zero_padding=True)|^2 as fp32 (utils/Forward_model.py:20-24,:39).

    When a gradient may be needed the propagated field U is saved (complex64, 8 B/pixel) so that the backward
    is one adjoint propagation of g = 2 w U (plus one derivative propagation if the distance needs a gradient).
    """

    @staticmethod
    def forward(ctx, amplitude, phase, z, lamb, px, phase_normalize, pad, band_limit=False):
        b, c, n = _check_field(phase, "phase")
        a, ph, in_mode = _amp_phase(amplitude, phase)
        zt, zd = prepare_distance(z, b, ph.device)
        need = any(ctx.needs_input_grad[:3])
        out = torch.empty((b, c, n, n), dtype=torch.float32, device=ph.device)
        u = torch.empty((b, c, n, n), dtype=torch.complex64, device=ph.device) if need else None
        _forward_call(a, ph, zt, zd, out, u, b, c, n, pad, in_mode, L.OUT_INTENSITY, lamb, px, phase_normalize, 1.0,
                      band_limit)
        if need:
            ctx.save_for_backward(a, ph, zt, u)
        ctx.meta = (b, c, n, bool(pad), float(lamb), float(px), zd, float(phase_normalize), amplitude.dtype, phase.dtype,
                    _z_meta(z), in_mode, tuple(amplitude.shape), bool(band_limit))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        a, ph, zt, u = ctx.saved_tensors
        b, c, n, pad, lamb, px, zd, pn, adt, pdt, z_meta, in_mode, ashape, bl = ctx.meta
        w = _f32(grad_out)
        ga = gp = gz = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            af = a if in_mode == L.IN_AMP_PHASE else a.expand(ph.shape).contiguous()
            ga = torch.empty_like(af)
            gp = torch.empty_like(ph)
            _adjoint_call(w, u, zt, zd, af, ph, ga, gp, b, c, n, pad, L.IN_COT_FIELD, L.OUT_GRAD_AP, lamb, px, pn, bl)
            ga = (ga if in_mode == L.IN_AMP_PHASE else ga.sum().reshape(ashape)).to(adt)
            gp = gp.to(pdt)
        if ctx.needs_input_grad[2] and z_meta is not None:
            gz = _grad_like(_grad_z_call(a, ph, zt, zd, w, u, L.IN_COT_FIELD, b, c, n, pad, in_mode, lamb, px, pn, bl),
                            z_meta)
        return ga, gp, gz, None, None, None, None, None


# ---------------------------------------------------------------------------------------------------
# fused no-grad fast paths
# ---------------------------------------------------------------------------------------------------
def holo_abs_angle(amplitude, phase, z, lamb, px, phase_normalize, pad=True, band_limit=False):
    """(|U|, angle U) in one pipeline (utils/Forward_model.py:27-34), no autograd graph."""
    b, c, n = _check_field(phase, "phase")
    a, ph, in_mode = _amp_phase(amplitude, phase)
    zt, zd = prepare_distance(z, b, ph.device)
    amp = torch.empty((b, c, n, n), dtype=torch.float32, device=ph.device)
    ang = torch.empty_like(amp)
    _forward_call(a, ph, zt, zd, amp, ang, b, c, n, pad, in_mode, L.OUT_ABS_ANGLE, lamb, px, phase_normalize, 1.0,
                  band_limit)
    return amp, ang


def holo_intensity_pair(amplitude, phase_a, phase_b, z_a, z_b, lamb, px, phase_normalize, pad=True, band_limit=False):
    """Two no-grad intensity syntheses sharing one amplitude (utils/Data_loader.py:31-32) written into ONE [2B,C,N,N]
    output allocation, without concatenating the inputs: each phase tensor is read in place."""
    b, c, n = _check_field(phase_a, "phase")
    out = torch.empty((2 * b, c, n, n), dtype=torch.float32, device=phase_a.device)
    for k, (ph_k, z_k) in enumerate(((phase_a, z_a), (phase_b, z_b))):
        a, ph, in_mode = _amp_phase(amplitude, ph_k)
        zt, zd = prepare_distance(z_k, b, ph.device)
        _forward_call(a, ph, zt, zd, out[k * b:(k + 1) * b], None, b, c, n, pad, in_mode, L.OUT_INTENSITY, lamb, px,
                      phase_normalize, 1.0, band_limit)
    return out[:b], out[b:]


def back_prop_fused(holo, z, lamb, px, amplitude_normalize, amp_pha: bool, band_limit: bool = False):
    """cat(|s U|, angle(s U)) or cat(re, im) * s of U = ASM(sqrt(holo), z) in one pipeline
    (utils/Forward_model.py:55-65), fp32 [B,2,N,N]."""
    b, c, n = _check_field(holo, "holo")
    if c != 1:
        raise RuntimeError("Back_prop expects single-channel holograms [B,1,N,N]")
    if holo.is_complex():
        raise RuntimeError("Back_prop expects a real hologram")
    h = _f32(holo)
    zt, zd = prepare_distance(z, b, h.device)
    out = torch.empty((b, 2, n, n), dtype=torch.float32, device=h.device)
    _forward_call(h, None, zt, zd, out, None, b, 1, n, False, L.IN_SQRT_REAL,
                  L.OUT_ABSANG_CAT if amp_pha else L.OUT_REIM_CAT, lamb, px, 1.0, amplitude_normalize, band_limit)
    return out


def unwrap_phase(x: torch.Tensor) -> torch.Tensor:
    """Device-side 2-D phase unwrapping (``asm_b200_unwrap``, include/asm_b200.h); see ``Forward_model.unwrap``."""
    if not isinstance(x, torch.Tensor) or not x.is_cuda:
        raise RuntimeError("unwrap_phase needs a CUDA tensor (no CPU fallback)")
    if x.dim() == 4 and x.shape[1] == 1:
        b, h, w = x.shape[0], x.shape[2], x.shape[3]
    elif x.dim() == 3:
        b, h, w = x.shape
    elif x.dim() == 2:
        b, (h, w) = 1, x.shape
    else:
        raise RuntimeError("unwrap_phase expects [B, 1, H, W], [B, H, W] or [H, W]")
    lib = L.load()
    need = lib.asm_b200_unwrap_workspace_bytes(b, h, w)
    if need == 0:
        raise RuntimeError(f"unwrap_phase: unsupported shape {tuple(x.shape)} "
                           "(H, W >= 3, H W <= 2^28, B (2 H W - H - W) <= 2^31 - 1)")
    ph = x.detach().to(torch.float32).contiguous()
    out = torch.empty((b, 1, h, w), dtype=torch.float32, device=x.device)
    with torch.cuda.device(x.device):
        ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        L.check(lib.asm_b200_unwrap(ph.data_ptr(), out.data_ptr(), b, h, w, ws.data_ptr(), need,
                                    torch.cuda.current_stream().cuda_stream))
    return out
