"""GPU: the transfer function of every kernel family, bin by bin.

A unit impulse at (0, 0) propagated without padding comes out as ifft2(H), so a float64 fft2 of the kernel's output
recovers the H the kernel applied on all M^2 bins; it must match oracle.asm_oracle.transfer_function to TOL_H on every
bin.  This sees what a rel-L2 bound over a whole field cannot: one wrong bin, one wrong row (the folded kappa tables,
the digit-reversed column orders, the separately staged Nyquist row), and the evanescent clamp (H = 1 there) of every
table builder, in three optics: none, a ring (~9 %) and most (~69 %) of the bins evanescent.
"""
import numpy as np
import pytest
import torch

from oracle import asm_oracle as ao
from _parity import (OPTICS, abi_adjoint, abi_forward, assert_well_conditioned, check_transfer, empty_device,
                     evanescent_fraction, recover_h, to_device)

pytestmark = pytest.mark.gpu

Z32 = np.array([6e-3, -20e-3], dtype=np.float32)
Z64 = np.array([0.0123456789, 0.5], dtype=np.float64)   # |z| < 2 m: the double-float phase's range (k32t.cuh)
ZMAX = 0.5


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as p
    p._lib.load()
    return p


# FFT families (generic <= 512, k32t 1024, k64 2048, on-the-fly H at 4096) and the matrix-product path (other N)
SIZES = [32, 64, 128, 256, 512, 1024, 2048, 4096, 45, 92, 250, 1000]
CASES = [(n, o) for n in SIZES for o in OPTICS]

# (operation, in_mode, input offset, output offset, z): the bulk (aligned) and register (offset by one element) row
# kernels on both sides, real input, and the adjoint (conj(H)).  Samples carry different z, and C = 2 channels each.
VARIANTS = [("fwd", ao.IN_COMPLEX, 0, 0, Z32), ("fwd", ao.IN_COMPLEX, 1, 1, Z64), ("fwd", ao.IN_REAL, 0, 0, Z64),
            ("fwd", ao.IN_REAL, 1, 0, Z32), ("adj", ao.IN_COMPLEX, 0, 0, Z64), ("adj", ao.IN_COMPLEX, 1, 1, Z32)]


def _run(pkg, op, in_mode, off_in, off_out, z, n, lamb, px, b=2, c=2):
    L = pkg._lib
    if in_mode == ao.IN_COMPLEX:
        imp = np.zeros((b, c, n, n), dtype=np.complex64)
    else:
        imp = np.zeros((b, c, n, n), dtype=np.float32)
    imp[:, :, 0, 0] = 1.0
    x = to_device(imp, off_in)
    zt = torch.from_numpy(z).cuda()
    out = empty_device((b, c, n, n), torch.complex64, off_out)
    if op == "fwd":
        abi_forward(L, x, None, zt, out, None, b, c, n, 0, in_mode, ao.OUT_COMPLEX, lamb, px)
    else:
        abi_adjoint(L, x, None, zt, None, None, out, None, b, c, n, 0, in_mode, ao.OUT_COMPLEX, lamb, px)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("n,optics", CASES, ids=[f"{n}-{o}" for n, o in CASES])
def test_transfer_function_per_bin(pkg, n, optics):
    lamb, px = OPTICS[optics]
    worst_phase = assert_well_conditioned(n, n, lamb, px, ZMAX)
    print(f"\nM={n} {optics}: {100 * evanescent_fraction(n, n, lamb, px):.1f} % evanescent, "
          f"phase change of one rounding of arg <= {worst_phase:.1e} rad")
    worst = 0.0
    for op, in_mode, off_in, off_out, z in VARIANTS:
        h_ref = ao.transfer_function(n, n, lamb, px, z)
        if op == "adj":
            h_ref = np.conj(h_ref)
        h = recover_h(_run(pkg, op, in_mode, off_in, off_out, z, n, lamb, px))
        for c in range(h.shape[1]):
            worst = max(worst, check_transfer(h[:, c], h_ref, f"{op} in{in_mode} off({off_in},{off_out}) "
                                                               f"{z.dtype} channel {c}"))
    print(f"M={n} {optics}: worst per-bin |dH| = {worst:.3e}")


@pytest.mark.parametrize("n,moments", [(n, m) for n in (1024, 2048, 4096, 92) for m in (False, True)])
def test_focal_stack_per_bin(pkg, n, moments):
    """The focal stack's out-of-place column pass (k32t_lines, k64_cols, k_cols) and its moment-writing inverse row
    kernels, ring optics: every plane's H bin by bin, and the moments against those of the oracle's planes."""
    lamb, px = OPTICS["ring"]
    assert_well_conditioned(n, n, lamb, px, ZMAX)
    b, k = (1, 2) if n >= 4096 else (2, 3)
    zz = np.array([[6e-3, -20e-3, 0.0123456789], [0.5, -3e-3, 1e-4]])[:b, :k]
    z = zz.astype(np.float64 if moments else np.float32)
    imp = np.zeros((b, n, n), dtype=np.complex64)
    imp[:, 0, 0] = 1.0
    res = pkg.focal_stack(torch.from_numpy(imp).cuda(), torch.from_numpy(z).cuda(), lamb, px, output="complex",
                          moments=moments)
    u, mom = res if moments else (res, None)
    torch.cuda.synchronize()
    u = u.cpu().numpy()
    h = recover_h(u)
    h_ref = ao.transfer_function(n, n, lamb, px, z.reshape(-1)).reshape(b, k, n, n)
    check_transfer(h, h_ref, f"focal stack N={n} moments={moments}")
    if moments:
        a = np.abs(np.fft.ifft2(h_ref)).reshape(b, k, -1)
        mref = np.stack([a.sum(-1), (a ** 2).sum(-1), (a ** 4).sum(-1)], axis=-1)
        rel = np.abs(mom.cpu().numpy() - mref) / mref
        print(f"  moments: max rel err {rel.max():.3e}")
        assert rel.max() < 1e-5, rel.max()
