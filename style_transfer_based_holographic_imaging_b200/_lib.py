"""ctypes binding of the C ABI in include/asm_b200.h.  No CPU fallback: if the CUDA library is missing or
cannot be loaded, importing the product path raises."""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ASM_B200_LIB", os.path.join(HERE, "libasm_b200.so"))   # override: A/B testing of build variants

# mode constants (mirror include/asm_b200.h)
Z_F32, Z_F64 = 0, 1
IN_COMPLEX, IN_AMP_PHASE, IN_SQRT_REAL, IN_COT_FIELD, IN_REAL, IN_CONST_AMP_PHASE = 0, 1, 2, 3, 4, 5
OUT_COMPLEX, OUT_INTENSITY, OUT_ABS_ANGLE, OUT_REIM_CAT, OUT_ABSANG_CAT, OUT_GRAD_AP = 0, 1, 2, 3, 4, 5
ABI_VERSION = 1

SYMBOLS = ["asm_b200_abi_version", "asm_b200_strerror", "asm_b200_workspace_bytes", "asm_b200_forward",
           "asm_b200_adjoint", "asm_b200_grad_z", "asm_b200_launch_count", "asm_b200_profile",
           "asm_b200_unwrap_workspace_bytes", "asm_b200_unwrap", "asm_b200_focal_stack_workspace_bytes",
           "asm_b200_focal_stack"]

_lib = None


class AsmB200Error(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise AsmB200Error(
            f"{LIB_PATH} is missing: build it with `python -m style_transfer_based_holographic_imaging_b200.build` "
            "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    vp, ci, cd, cf, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_float, ctypes.c_size_t
    lib.asm_b200_abi_version.restype = ci
    lib.asm_b200_abi_version.argtypes = []
    lib.asm_b200_strerror.restype = ctypes.c_char_p
    lib.asm_b200_strerror.argtypes = [ci]
    lib.asm_b200_workspace_bytes.restype = sz
    lib.asm_b200_workspace_bytes.argtypes = [ci, ci, ci, ci]
    lib.asm_b200_forward.restype = ci
    lib.asm_b200_forward.argtypes = [vp, vp, vp, ci, vp, vp, ci, ci, ci, ci, ci, ci, cd, cd, cf, cf, vp, sz, vp]
    lib.asm_b200_adjoint.restype = ci
    lib.asm_b200_adjoint.argtypes = [vp, vp, vp, ci, vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, cd, cd, cf, vp, sz, vp]
    lib.asm_b200_grad_z.restype = ci
    lib.asm_b200_grad_z.argtypes = [vp, vp, vp, ci, vp, vp, ci, vp, ci, ci, ci, ci, ci, cd, cd, cf, vp, sz, vp]
    lib.asm_b200_launch_count.restype = ctypes.c_ulonglong
    lib.asm_b200_launch_count.argtypes = []
    lib.asm_b200_profile.restype = None
    lib.asm_b200_profile.argtypes = [ci, ctypes.POINTER(ctypes.c_double)]
    lib.asm_b200_unwrap_workspace_bytes.restype = sz
    lib.asm_b200_unwrap_workspace_bytes.argtypes = [ci, ci, ci]
    lib.asm_b200_unwrap.restype = ci
    lib.asm_b200_unwrap.argtypes = [vp, vp, ci, ci, ci, vp, sz, vp]
    lib.asm_b200_focal_stack_workspace_bytes.restype = sz
    lib.asm_b200_focal_stack_workspace_bytes.argtypes = [ci, ci, ci, ci]
    lib.asm_b200_focal_stack.restype = ci
    lib.asm_b200_focal_stack.argtypes = [vp, vp, vp, ci, ci, vp, vp, vp, ci, ci, ci, ci, ci, cd, cd, cf, vp, sz, vp]
    if lib.asm_b200_abi_version() != ABI_VERSION:
        raise AsmB200Error("libasm_b200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise AsmB200Error(load().asm_b200_strerror(rc).decode())
