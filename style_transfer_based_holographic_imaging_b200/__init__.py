"""B200-native (sm_100a) angular-spectrum propagation for holographic imaging.

Drop-in for the hot path of csleemooo/style_transfer_based_holographic_imaging:
``ASM`` (utils/Angular_Spectrum_Method.py), ``Holo_Generator`` / ``Back_prop`` (utils/Forward_model.py) and the
backward autograd derives from them.  The compute path is ``libasm_b200.so`` (hand-written CUDA behind the C
ABI in include/asm_b200.h); this package is the host-side mirror of the reference interface.
"""
from . import _lib
from .Angular_Spectrum_Method import ASM, torch_fft, torch_ifft, center_crop
from .Forward_model import Holo_Generator, Back_prop, unwrap
from .functional import asm_forward_raw, asm_adjoint_raw, AsmPropagate, HoloIntensity, HoloField
from .focus import focal_stack, focus_metric, autofocus

__all__ = ["ASM", "Holo_Generator", "Back_prop", "torch_fft", "torch_ifft", "center_crop",
           "asm_forward_raw", "asm_adjoint_raw", "AsmPropagate", "HoloIntensity", "HoloField", "unwrap",
           "focal_stack", "focus_metric", "autofocus"]
