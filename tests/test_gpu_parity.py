"""GPU parity tests (-m gpu): the CUDA path, called through the drop-in Python interface (which goes through
the C ABI of include/asm_b200.h), against the oracle and the committed golden vectors.

Tolerance: BASELINE.json north_star -- 1e-4 relative L2 in fp32.  The oracle runs in float64, so what is
measured is the kernel's own fp32 error (~3e-7); TOL below is the contract, per-shape errors are printed.
"""
import numpy as np
import pytest
import torch

from oracle import asm_oracle as ao
from oracle.make_golden import at

pytestmark = pytest.mark.gpu

TOL = 1e-4          # north_star contract
TOL_GRAD = 1e-4
LAMB, PX = 532e-9, 1.5e-6


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as m
    m._lib.load()   # fail loudly if the CUDA library is not there
    return m


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _field(rng, b, n):
    return (rng.standard_normal((b, 1, n, n)) + 1j * rng.standard_normal((b, 1, n, n))).astype(np.complex64)


@pytest.mark.parametrize("n,pad", [(32, False), (32, True), (64, False), (64, True), (128, False), (128, True),
                                   (256, False), (256, True), (512, False), (512, True), (1024, False), (16, True)])
def test_asm_forward_vs_oracle(pkg, n, pad):
    rng = np.random.default_rng(100 + n + int(pad))
    b = 3 if n <= 256 else 2
    O = _field(rng, b, n)
    d = ((0.2 + 0.8 * rng.random((b, 1, 1, 1))) * 6e-3).astype(np.float32)
    with torch.no_grad():
        U = pkg.ASM(_dev(O), LAMB, _dev(d), PX, zero_padding=pad)
    assert U.dtype == torch.complex64 and tuple(U.shape) == (b, 1, n, n)
    err = ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, d, PX, pad))
    print(f"ASM N={n} pad={pad}: rel-L2 {err:.3e}")
    assert err < TOL


@pytest.mark.parametrize("n,pad", [(1024, True), (2048, False), (2048, True), (4096, False)])
def test_asm_forward_large_vs_oracle(pkg, n, pad):
    rng = np.random.default_rng(n + int(pad))
    O = _field(rng, 1, n)
    d = np.array([[[[7.3e-3]]]], dtype=np.float32)
    with torch.no_grad():
        U = pkg.ASM(_dev(O), LAMB, _dev(d), PX, zero_padding=pad)
    err = ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, d, PX, pad))
    print(f"ASM N={n} pad={pad}: rel-L2 {err:.3e}")
    assert err < TOL


@pytest.mark.parametrize("n,pad", [(64, False), (64, True), (256, False), (256, True), (1024, False), (512, True)])
def test_adjoint_vs_oracle_and_dot_product(pkg, n, pad):
    rng = np.random.default_rng(7 * n + int(pad))
    b = 2
    x, y = _field(rng, b, n), _field(rng, b, n)
    d = ((0.2 + 0.8 * rng.random((b, 1, 1, 1))) * 3e-3).astype(np.float32)
    zx = _dev(d)
    aty = pkg.asm_adjoint_raw(_dev(y), zx, LAMB, PX, pad)
    err = ao.rel_l2(aty.cpu().numpy(), ao.asm_adjoint(y, LAMB, d, PX, pad))
    print(f"adjoint N={n} pad={pad}: rel-L2 {err:.3e}")
    assert err < TOL
    ax = pkg.asm_forward_raw(_dev(x), zx, LAMB, PX, pad)
    lhs = torch.vdot(_dev(y).flatten().to(torch.complex128), ax.flatten().to(torch.complex128))
    rhs = torch.vdot(aty.flatten().to(torch.complex128), _dev(x).flatten().to(torch.complex128))
    assert abs(lhs - rhs).item() < 1e-5 * abs(lhs).item()


ASM_CASES = ["asm_n32", "asm_n32_pad", "asm_n64_far", "asm_n64_pad_far", "asm_n64_evan", "asm_n32_pad_evan",
             "asm_n128_neg", "asm_n128_pad"]


@pytest.mark.parametrize("name", ASM_CASES)
def test_asm_reference_vectors_and_autograd(pkg, ref_cases, name):
    """Outputs and gradients of the reference itself (tests/golden/ref_cases.npz, oracle/make_golden.py)."""
    c = ref_cases
    B, N, pad, lamb, px = c[f"{name}.meta"]
    pad = bool(pad)
    O = _dev(c[f"{name}.O"]).requires_grad_(True)
    d = _dev(c[f"{name}.d"]).requires_grad_(True)
    G = _dev(c[f"{name}.G"])
    ix = c[f"{name}.idx"]
    U = pkg.ASM(O, float(lamb), d, float(px), zero_padding=pad)
    e_u = ao.rel_l2(at(U.detach().cpu().numpy(), ix), c[f"{name}.U"])
    L = torch.real(torch.sum(torch.conj(G) * U))
    gO, gd = torch.autograd.grad(L, [O, d])
    e_go = ao.rel_l2(at(gO.cpu().numpy(), ix), c[f"{name}.gO"])
    e_gd = ao.rel_l2(gd.cpu().numpy(), c[f"{name}.gd"])
    print(f"{name}: U {e_u:.3e}  grad_O {e_go:.3e}  grad_d {e_gd:.3e}")
    assert e_u < TOL and e_go < TOL_GRAD and e_gd < TOL_GRAD
    assert gd.shape == d.shape and gd.dtype == d.dtype


def _args(**kw):
    return ao.Optics(**kw)


def test_mnist_bundled_holograms(pkg, mnist_golden):
    """The reference's own fixtures (test_data/*.pt): Holo_Generator intensity, all 20 x 5 samples, each at the stored
    sample of its pixels."""
    g = mnist_golden
    hg = pkg.Holo_Generator(_args()).cuda()
    worst = 0.0
    for i in range(g["gt_phase"].shape[0]):
        ph = _dev(g["gt_phase"][i])
        amp = torch.full_like(ph, float(g["amplitude"]))
        with torch.no_grad():
            holo = hg(amp, ph, _dev(g["distance_content"][i]))
        assert holo.dtype == torch.float32
        for j in range(holo.shape[0]):
            worst = max(worst, ao.rel_l2(holo[j].cpu().numpy().reshape(-1)[g["holo_idx"]], g["content_holo"][i][j]))
    print(f"MNIST bundled holograms (N=128, FFT 256): worst rel-L2 {worst:.3e}")
    assert worst < TOL


@pytest.mark.parametrize("name", ["hg_n32", "hg_n64_norm", "hg_n128_neg"])
def test_holo_generator_reference_vectors(pkg, ref_cases, name):
    c = ref_cases
    B, N, lamb, px, pn, dn, dc = c[f"{name}.meta"]
    hg = pkg.Holo_Generator(_args(wavelength=lamb, pixel_size=px, phase_normalize=pn, distance_normalize=dn,
                                  distance_normalize_constant=dc))
    A = _dev(c[f"{name}.A"]).requires_grad_(True)
    P = _dev(c[f"{name}.P"]).requires_grad_(True)
    d = _dev(c[f"{name}.d"]).requires_grad_(True)
    ix = c[f"{name}.idx"]
    I = hg(A, P, d)
    assert I.dtype == torch.float32
    e_i = ao.rel_l2(at(I.detach().cpu().numpy(), ix), c[f"{name}.I"])
    gA, gP, gd = torch.autograd.grad(torch.sum(_dev(c[f"{name}.W"]) * I), [A, P, d])
    e_a, e_p, e_d = (ao.rel_l2(at(gA.cpu().numpy(), ix), c[f"{name}.gA"]), ao.rel_l2(at(gP.cpu().numpy(), ix), c[f"{name}.gP"]),
                     ao.rel_l2(gd.cpu().numpy(), c[f"{name}.gd"]))
    print(f"{name}: I {e_i:.3e} grad_A {e_a:.3e} grad_phase {e_p:.3e} grad_d {e_d:.3e}")
    assert e_i < TOL and e_a < TOL_GRAD and e_p < TOL_GRAD and e_d < TOL_GRAD
    with torch.no_grad():
        amp, ph = hg(A, P, d, return_field=True)
        U = hg(A, P, d, complex_number=True)
    assert ao.rel_l2(at(amp.cpu().numpy(), ix), c[f"{name}.amp"]) < TOL
    assert ao.rel_l2(np.exp(1j * at(ph.cpu().numpy(), ix).astype(np.float64)), np.exp(1j * c[f"{name}.ph"].astype(np.float64))) < TOL
    assert ao.rel_l2(at(U.cpu().numpy(), ix), c[f"{name}.U"]) < TOL
    # gradients through the (abs, angle) outputs
    a2, p2 = hg(A, P, d, return_field=True)
    gA2, gP2, gd2 = torch.autograd.grad(torch.sum(_dev(c[f"{name}.Wa"]) * a2) + torch.sum(_dev(c[f"{name}.Wp"]) * p2), [A, P, d])
    assert ao.rel_l2(at(gA2.cpu().numpy(), ix), c[f"{name}.gA2"]) < 5e-4
    assert ao.rel_l2(at(gP2.cpu().numpy(), ix), c[f"{name}.gP2"]) < 5e-4
    assert ao.rel_l2(gd2.cpu().numpy(), c[f"{name}.gd2"]) < 5e-4


@pytest.mark.parametrize("name", ["bp_n64_amp_pha", "bp_n64_re_im", "bp_n32_amp_pha"])
def test_back_prop_reference_vectors(pkg, ref_cases, name):
    c = ref_cases
    B, N, an, amp_pha = c[f"{name}.meta"]
    bp = pkg.Back_prop(_args(amplitude_normalize=float(an), Holo_G_input="amp_pha" if amp_pha else "real_imag"))
    with torch.no_grad():
        out = bp(_dev(c[f"{name}.holo"]), _dev(c[f"{name}.d"])).cpu().numpy()
    assert out.shape == (int(B), 2, int(N), int(N))
    out, ref = at(out, c[f"{name}.idx"]), c[f"{name}.out"]      # one row per channel
    if amp_pha:
        assert ao.rel_l2(out[0], ref[0]) < TOL
        assert ao.rel_l2(np.exp(1j * out[1].astype(np.float64)), np.exp(1j * ref[1].astype(np.float64))) < TOL
    else:
        assert ao.rel_l2(out, ref) < TOL


def test_distance_argument_forms(pkg):
    """python float / 0-dim / fp64 distances follow the reference's dtype rules for the phase constant."""
    rng = np.random.default_rng(5)
    O = _field(rng, 2, 64)
    x = _dev(O)
    for d, dn in [(0.0031, np.float64(0.0031)), (torch.tensor(0.0031).cuda(), np.float32(0.0031)),
                  (torch.tensor(0.0031, dtype=torch.float64).cuda(), np.float64(0.0031))]:
        with torch.no_grad():
            U = pkg.ASM(x, LAMB, d, PX)
        assert ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, dn, PX)) < 2e-6   # fp32-vs-fp64 constant differs by ~5e-5


@pytest.mark.parametrize("n,pad", [(1024, False), (512, True), (2048, False)])
def test_fp64_distances_double_float_phase(pkg, n, pad):
    """fp64 / python-float distances on the double-float H of the FFT-1024 / FFT-2048 paths: the phase constant 2 pi z is
    not an fp32 number there, so the (hi, lo) split of c is exercised (csrc/k32t.cuh, k64.cuh); forward, adjoint and the
    distance gradient, at a far distance."""
    rng = np.random.default_rng(n + int(pad))
    O, G = _field(rng, 1, n), _field(rng, 1, n)
    x, g = _dev(O), _dev(G)
    for d in (0.0123456789, -0.0199):
        dn = np.float64(d)
        with torch.no_grad():
            U = pkg.ASM(x, LAMB, d, PX, zero_padding=pad)
            A = pkg.asm_adjoint_raw(g, torch.tensor([d], dtype=torch.float64).cuda(), LAMB, PX, pad)
        e_u = ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, dn, PX, pad))
        e_a = ao.rel_l2(A.cpu().numpy(), ao.asm_adjoint(G, LAMB, dn, PX, pad))
        print(f"n={n} pad={pad} z={d}: forward {e_u:.2e} adjoint {e_a:.2e}")
        assert e_u < 2e-6 and e_a < 2e-6
    # distance gradient through the complex field with an fp64 distance tensor
    dt = torch.tensor([[[[0.0123456789]]]], dtype=torch.float64).cuda().requires_grad_(True)
    U = pkg.ASM(x, LAMB, dt, PX, zero_padding=pad)
    (gd,) = torch.autograd.grad(torch.real(torch.sum(torch.conj(g) * U)), [dt])
    eps = 1e-9                                                     # 2 pi eps / lambda = 0.012 rad: central differences hold
    up = ao.asm(O, LAMB, np.float64(0.0123456789 + eps), PX, pad)
    um = ao.asm(O, LAMB, np.float64(0.0123456789 - eps), PX, pad)
    fd = np.real(np.sum(np.conj(G) * (up - um))) / (2 * eps)
    assert abs(gd.item() - fd) < 2e-3 * abs(fd), (gd.item(), fd)


def test_multichannel_broadcast(pkg):
    rng = np.random.default_rng(9)
    O = (rng.standard_normal((2, 3, 64, 64)) + 1j * rng.standard_normal((2, 3, 64, 64))).astype(np.complex64)
    d = np.array([4e-4, 9e-4], dtype=np.float32).reshape(2, 1, 1, 1)
    with torch.no_grad():
        U = pkg.ASM(_dev(O), LAMB, _dev(d), PX, zero_padding=True)
    assert ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, d, PX, True)) < TOL


def test_errors(pkg):
    z = torch.tensor([[[[1e-3]]]]).cuda()
    with pytest.raises(RuntimeError):
        pkg.ASM(torch.zeros(1, 1, 64, 64, dtype=torch.complex64), LAMB, 1e-3, PX)            # CPU tensor
    with pytest.raises(RuntimeError):
        pkg.ASM(torch.zeros(1, 1, 64, 32, dtype=torch.complex64).cuda(), LAMB, z, PX)        # non-square
    with pytest.raises(RuntimeError):
        pkg.ASM(torch.zeros(1, 1, 49, 49, dtype=torch.complex64).cuda(), LAMB, z, PX, zero_padding=True)   # odd N with padding (the reference raises too)
    with pytest.raises(RuntimeError):
        pkg.ASM(torch.zeros(2, 1, 64, 64, dtype=torch.complex64).cuda(), LAMB, torch.zeros(3).cuda(), PX)  # bad d shape


@pytest.mark.parametrize("n,b", [(1024, 48), (256, 512)])
def test_full_size_properties(pkg, n, b):
    """Size-independent properties at bench-scale batches: unitarity (|H| = 1, no evanescent bins at the default
    optics), linearity, and batch independence (a sample's result does not depend on its chunk)."""
    g = torch.Generator(device="cuda").manual_seed(1)
    O = torch.randn(b, 1, n, n, 2, device="cuda", generator=g)
    O = torch.view_as_complex(O)
    z = (0.2 + 0.8 * torch.rand(b, 1, 1, 1, device="cuda", generator=g)) * 6e-3
    U = pkg.asm_forward_raw(O, z, LAMB, PX, False)
    e_in = (O.abs() ** 2).sum(dim=(1, 2, 3), dtype=torch.float64)
    e_out = (U.abs() ** 2).sum(dim=(1, 2, 3), dtype=torch.float64)
    assert torch.max(torch.abs(e_out / e_in - 1)).item() < 1e-5
    # fwd then adjoint is the identity for a unitary operator
    back = pkg.asm_adjoint_raw(U, z, LAMB, PX, False)
    assert (torch.linalg.vector_norm(back - O) / torch.linalg.vector_norm(O)).item() < 1e-5
    # batch independence, bitwise
    idx = [0, b // 2, b - 1]
    Us = pkg.asm_forward_raw(O[idx].contiguous(), z[idx].contiguous(), LAMB, PX, False)
    assert torch.equal(Us, U[idx])
    # linearity
    U2 = pkg.asm_forward_raw(2.5 * O[:4], z[:4], LAMB, PX, False)
    assert (torch.linalg.vector_norm(U2 - 2.5 * U[:4]) / torch.linalg.vector_norm(U2)).item() < 1e-6


def test_physics_loss_training_step_decreases_loss(pkg):
    """SURVEY 8(f) row 1: the drop-in forward model inside an optimisation loop with a learned distance
    (gradients w.r.t. amplitude, phase and d all flow through the CUDA path)."""
    torch.manual_seed(0)
    hg = pkg.Holo_Generator(_args())
    n, b = 64, 4
    gt_ph = torch.rand(b, 1, n, n, device="cuda")
    gt_amp = torch.full_like(gt_ph, 0.6)
    d_true = torch.tensor([0.45, 0.5, 0.6, 0.7], device="cuda").view(b, 1, 1, 1)
    with torch.no_grad():
        target = hg(gt_amp, gt_ph, d_true)
    amp = torch.full_like(gt_ph, 0.5).requires_grad_(True)
    # (a constant start field is a plane wave: |U|^2 does not depend on d and grad_d is exactly 0, so start textured)
    ph = (0.2 * torch.rand_like(gt_ph)).requires_grad_(True)
    d = (d_true + 0.03).clone().requires_grad_(True)
    opt = torch.optim.Adam([amp, ph, d], lr=2e-2)
    losses = []
    for _ in range(60):
        loss = torch.mean((hg(amp, ph, d) - target) ** 2)
        opt.zero_grad()
        loss.backward()
        assert d.grad is not None and torch.isfinite(d.grad).all() and d.grad.abs().sum() > 0
        opt.step()
        losses.append(loss.item())
    assert losses[-1] < 0.3 * losses[0], (losses[0], losses[-1])


def test_edge_cases(pkg):
    """z = 0 is the identity, far and negative distances, single sample, non-contiguous views, fp64 inputs,
    gradient for the distance only, and unwrap=True on the device."""
    rng = np.random.default_rng(21)
    O = _field(rng, 1, 64)
    x = _dev(O)
    U0 = pkg.ASM(x, LAMB, torch.zeros(1, 1, 1, 1, device="cuda"), PX)
    assert ao.rel_l2(U0.cpu().numpy(), O) < 1e-6                        # H = 1
    for zval in (20e-3, -20e-3):                                         # theta up to 2.4e5 rad
        d = np.full((1, 1, 1, 1), zval, dtype=np.float32)
        U = pkg.ASM(x, LAMB, _dev(d), PX, zero_padding=True)
        assert ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, d, PX, True)) < TOL
    # non-contiguous input view and fp64 amplitude / phase
    big = _dev(_field(rng, 2, 128))
    view = big[:, :, ::2, ::2]
    assert not view.is_contiguous()
    d2 = np.array([3e-4, 5e-4], dtype=np.float32).reshape(2, 1, 1, 1)
    U = pkg.ASM(view, LAMB, _dev(d2), PX)
    assert ao.rel_l2(U.cpu().numpy(), ao.asm(view.cpu().numpy(), LAMB, d2, PX)) < TOL
    hg = pkg.Holo_Generator(_args())
    A = torch.rand(2, 1, 64, 64, device="cuda", dtype=torch.float64)
    P = torch.rand(2, 1, 64, 64, device="cuda", dtype=torch.float64)
    dn = torch.tensor([0.5, 0.7], device="cuda").view(2, 1, 1, 1)
    I = hg(A, P, dn)
    assert I.dtype == torch.float32
    assert ao.rel_l2(I.cpu().numpy(), ao.holo_generator(A.cpu().numpy(), P.cpu().numpy(), dn.cpu().numpy(), _args())) < TOL
    # gradient w.r.t. the distance only
    dq = dn.clone().requires_grad_(True)
    (gd,) = torch.autograd.grad(hg(A.float(), P.float(), dq).sum(), [dq])
    assert gd.shape == dq.shape and torch.isfinite(gd).all()
    # unwrap=True runs on the device (asm_b200_unwrap): amplitude untouched, phase moved by multiples of 2 pi only
    a_u, p_u = hg(A.float(), P.float(), dn, return_field=True, unwrap=True)
    a_w, p_w = hg(A.float(), P.float(), dn, return_field=True)
    assert torch.equal(a_u, a_w) and p_u.is_cuda
    k = ((p_u - p_w) / (2 * np.pi)).cpu().numpy()
    assert np.abs(k - np.round(k)).max() < 1e-4


def test_multichannel_intensity_and_grads(pkg):
    """C > 1: the distance broadcasts over channels (the reference broadcasts its [B,1,M,M] transfer function)."""
    rng = np.random.default_rng(33)
    b, c, n = 2, 3, 32
    amp = (0.5 + 0.5 * rng.random((b, c, n, n))).astype(np.float32)
    ph = rng.random((b, c, n, n)).astype(np.float32)
    d = np.array([0.4, 0.8], dtype=np.float32).reshape(b, 1, 1, 1)
    w = rng.standard_normal((b, c, n, n)).astype(np.float32)
    hg = pkg.Holo_Generator(_args())
    A, P, D = _dev(amp).requires_grad_(True), _dev(ph).requires_grad_(True), _dev(d).requires_grad_(True)
    I = hg(A, P, D)
    gA, gP, gD = torch.autograd.grad(torch.sum(_dev(w) * I), [A, P, D])
    ref_i = np.stack([ao.holo_generator(amp[:, k:k + 1], ph[:, k:k + 1], d, _args())[:, 0] for k in range(c)], axis=1)
    assert ao.rel_l2(I.detach().cpu().numpy(), ref_i) < TOL
    gd_ref = sum(ao.holo_generator_vjp(amp[:, k:k + 1], ph[:, k:k + 1], d, w[:, k:k + 1], _args())[2] for k in range(c))
    ga_ref = np.concatenate([ao.holo_generator_vjp(amp[:, k:k + 1], ph[:, k:k + 1], d, w[:, k:k + 1], _args())[0] for k in range(c)], axis=1)
    assert ao.rel_l2(gA.cpu().numpy(), ga_ref) < TOL_GRAD
    assert ao.rel_l2(gD.cpu().numpy().reshape(-1), gd_ref) < 1e-3


def test_fft1024_unaligned_buffers_fall_back(pkg):
    """FFT size 1024: the default row kernels move rows with TMA bulk copies, which need 16-byte aligned rows.  Buffers
    that are contiguous but only 8-byte aligned (a view starting one complex64 into a larger allocation) must take the
    register-landing kernels and give the same answers -- input and output, forward (intensity, complex) and adjoint."""
    from style_transfer_based_holographic_imaging_b200 import _lib as L
    rng = np.random.default_rng(77)
    for n, pad in [(1024, False), (512, True)]:
        b = 2
        O = _field(rng, b, n)
        d = ((0.2 + 0.8 * rng.random((b, 1, 1, 1))) * 4e-3).astype(np.float32)
        flat = torch.empty(b * n * n + 1, dtype=torch.complex64, device="cuda")
        x = flat[1:].view(b, 1, n, n)
        x.copy_(_dev(O))
        assert x.is_contiguous() and x.data_ptr() % 16 == 8
        oflat = torch.empty(b * n * n + 1, dtype=torch.complex64, device="cuda")
        out = oflat[1:].view(b, 1, n, n)
        z = _dev(d)
        ref_u = ao.asm(O, LAMB, d, PX, pad)
        U = pkg.asm_forward_raw(x, z, LAMB, PX, pad, out=out)
        assert U.data_ptr() == out.data_ptr()
        assert ao.rel_l2(U.cpu().numpy(), ref_u) < TOL
        iflat = torch.empty(b * n * n + 1, dtype=torch.float32, device="cuda")
        iout = iflat[1:].view(b, 1, n, n)                                 # 4-byte aligned only
        I = pkg.asm_forward_raw(x, z, LAMB, PX, pad, out_mode=L.OUT_INTENSITY, out=iout)
        assert ao.rel_l2(I.cpu().numpy(), np.abs(ref_u) ** 2) < TOL
        A = pkg.asm_adjoint_raw(x, z, LAMB, PX, pad, out=out)
        assert ao.rel_l2(A.cpu().numpy(), ao.asm_adjoint(O, LAMB, d, PX, pad)) < TOL
        # aligned input, same answers through the bulk-copy kernels
        U2 = pkg.asm_forward_raw(_dev(O), z, LAMB, PX, pad)
        assert ao.rel_l2(U2.cpu().numpy(), ref_u) < TOL


def test_hologram_synthesis_pair(pkg):
    """SURVEY 8(f) row 2: the loader pattern (Data_loader.py:24-32) -- constant amplitude 0.6, zero-padded MNIST-like
    phase, two distance lists -- as one fused launch sequence; identical to the two separate calls and to the oracle."""
    torch.manual_seed(3)
    hg = pkg.Holo_Generator(_args(distance_normalize=2.0, distance_normalize_constant=0.1))
    b = 5
    ph_a = torch.nn.functional.pad(torch.rand(b, 1, 64, 64, device="cuda"), (32, 32, 32, 32))
    ph_b = torch.nn.functional.pad(torch.rand(b, 1, 64, 64, device="cuda"), (32, 32, 32, 32))
    amp = torch.ones_like(ph_a) * 0.6
    d_a = -0.1 + torch.tensor([0.2, 0.4, 0.6, 0.8, 1.0], device="cuda").view(b, 1, 1, 1) / 2.0
    d_b = -0.1 + torch.tensor([0.3, 0.5, 0.7, 0.9, 1.1], device="cuda").view(b, 1, 1, 1) / 2.0
    ha, hb = hg.forward_pair(amp, ph_a, ph_b, d_a, d_b)
    assert ha.dtype == torch.float32 and not ha.requires_grad and ha.shape == ph_a.shape
    assert torch.equal(ha, hg(amp, ph_a, d_a)) and torch.equal(hb, hg(amp, ph_b, d_b))
    ref = ao.holo_generator(amp.cpu().numpy(), ph_b.cpu().numpy(), d_b.cpu().numpy(),
                            _args(distance_normalize=2.0, distance_normalize_constant=0.1))
    assert ao.rel_l2(hb.cpu().numpy(), ref) < TOL


def test_concurrent_host_threads_same_device(pkg):
    """Two host threads, two streams, one device: the shared lane streams are guarded by a per-device issue mutex, so
    concurrent calls give the same bits as the same calls made one after the other."""
    import threading
    rng = np.random.default_rng(5)
    n, b = 1024, 6
    xs = [_dev(_field(rng, b, n)) for _ in range(2)]
    zs = [_dev(((0.2 + 0.8 * rng.random((b, 1, 1, 1))) * 3e-3).astype(np.float32)) for _ in range(2)]
    ref = [pkg.asm_forward_raw(xs[i], zs[i], LAMB, PX, False).clone() for i in range(2)]
    torch.cuda.synchronize()
    outs, errs = [None, None], []

    def work(i):
        try:
            st = torch.cuda.Stream()
            with torch.cuda.stream(st):
                for _ in range(4):
                    outs[i] = pkg.asm_forward_raw(xs[i], zs[i], LAMB, PX, False)
            st.synchronize()
        except Exception as e:  # pragma: no cover
            errs.append(e)

    th = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errs, errs
    for i in range(2):
        assert torch.equal(outs[i], ref[i])


@pytest.mark.parametrize("n,pad", [(1024, False), (512, True)])
def test_fft1024_far_and_negative_distances(pkg, n, pad):
    """Bead-scale |z| = 20 mm (theta up to 2.4e5 rad, SURVEY Appendix A) and the back-focus sign on the FFT-1024
    kernels: the fp64 phase reduction must hold the 1e-4 contract where an fp32 phase fails by 60x."""
    rng = np.random.default_rng(91)
    O = _field(rng, 2, n)
    d = np.array([20e-3, -20e-3], dtype=np.float32).reshape(2, 1, 1, 1)
    U = pkg.ASM(_dev(O), LAMB, _dev(d), PX, zero_padding=pad)
    e = ao.rel_l2(U.cpu().numpy(), ao.asm(O, LAMB, d, PX, pad))
    print(f"n={n} pad={pad} |z|=20mm rel-L2 {e:.3e}")
    assert e < TOL
    A = pkg.asm_adjoint_raw(_dev(O), _dev(d), LAMB, PX, pad)
    assert ao.rel_l2(A.cpu().numpy(), ao.asm_adjoint(O, LAMB, d, PX, pad)) < TOL
