"""CPU: pin the oracle (oracle/asm_oracle.py) against the reference's golden vectors.

* tests/golden/mnist_holo.npz -- the reference's own bundled fixtures (test_data/*.pt): known-answer test
  for Holo_Generator intensity mode, all 100 samples (each hologram at a fixed sample of its pixels).
* tests/golden/ref_cases.npz  -- outputs/gradients of the reference imported live (oracle/make_golden.py), image-sized
  ones at a fixed sample of positions.
* when the reference checkout is mounted (build container), also a live comparison in float64.
Tolerances: the stored vectors were produced by the reference's fp32 forward FFT, so agreement is ~2e-7;
we assert 2e-6 (field/intensity) and 1e-5 (gradients, one more fp32 pass).
"""
import numpy as np
import pytest

from oracle import asm_oracle as ao
from oracle import ref_import
from oracle.make_golden import at

ASM_CASES = ["asm_n32", "asm_n32_pad", "asm_n64_far", "asm_n64_pad_far", "asm_n64_evan", "asm_n32_pad_evan",
             "asm_n128_neg", "asm_n128_pad"]
HG_CASES = ["hg_n32", "hg_n64_norm", "hg_n128_neg"]
BP_CASES = ["bp_n64_amp_pha", "bp_n64_re_im", "bp_n32_amp_pha"]


def test_mnist_known_answers(mnist_golden):
    g = mnist_golden
    args = ao.Optics()  # test_field_retrieval_mnist.py:56-60 defaults
    worst = 0.0
    for i in range(g["gt_phase"].shape[0]):
        amp = np.full_like(g["gt_phase"][i], g["amplitude"])
        holo = ao.holo_generator(amp, g["gt_phase"][i], g["distance_content"][i], args)
        for j in range(holo.shape[0]):
            worst = max(worst, ao.rel_l2(holo[j].reshape(-1)[g["holo_idx"]], g["content_holo"][i][j]))
    assert worst < 2e-6, worst


@pytest.mark.parametrize("name", ASM_CASES)
def test_asm_vs_reference_vectors(ref_cases, name):
    c = ref_cases
    B, N, pad, lamb, px = c[f"{name}.meta"]
    pad = bool(pad)
    ix = c[f"{name}.idx"]
    u = ao.asm(c[f"{name}.O"], lamb, c[f"{name}.d"], px, pad)
    assert ao.rel_l2(at(u, ix), c[f"{name}.U"]) < 2e-6
    assert ao.rel_l2(ao.asm_closed_form(c[f"{name}.O"], lamb, c[f"{name}.d"], px, pad), u) < 1e-12
    go = ao.asm_adjoint(c[f"{name}.G"], lamb, c[f"{name}.d"], px, pad)
    assert ao.rel_l2(at(go, ix), c[f"{name}.gO"]) < 1e-5
    gd = ao.asm_grad_d(c[f"{name}.O"], c[f"{name}.G"], lamb, c[f"{name}.d"], px, pad)
    assert ao.rel_l2(gd, c[f"{name}.gd"].reshape(-1)) < 1e-5


@pytest.mark.parametrize("name", HG_CASES)
def test_holo_generator_vs_reference_vectors(ref_cases, name):
    c = ref_cases
    B, N, lamb, px, pn, dn, dc = c[f"{name}.meta"]
    args = ao.Optics(lamb, px, pn, dn, dc)
    A, P, d, ix = c[f"{name}.A"], c[f"{name}.P"], c[f"{name}.d"], c[f"{name}.idx"]
    assert ao.rel_l2(at(ao.holo_generator(A, P, d, args), ix), c[f"{name}.I"]) < 2e-6
    amp, ph = ao.holo_generator(A, P, d, args, return_field=True)
    assert ao.rel_l2(at(amp, ix), c[f"{name}.amp"]) < 2e-6
    # compare phases on the unit circle (angle wraps at +-pi)
    assert ao.rel_l2(np.exp(1j * at(ph, ix).astype(np.float64)), np.exp(1j * c[f"{name}.ph"].astype(np.float64))) < 5e-6
    assert ao.rel_l2(at(ao.holo_generator(A, P, d, args, complex_number=True), ix), c[f"{name}.U"]) < 2e-6
    ga, gp, gd = ao.holo_generator_vjp(A, P, d, c[f"{name}.W"], args)
    assert ao.rel_l2(at(ga, ix), c[f"{name}.gA"]) < 1e-5
    assert ao.rel_l2(at(gp, ix), c[f"{name}.gP"]) < 1e-5
    assert ao.rel_l2(gd, c[f"{name}.gd"].reshape(-1)) < 1e-5


@pytest.mark.parametrize("name", BP_CASES)
def test_back_prop_vs_reference_vectors(ref_cases, name):
    c = ref_cases
    B, N, an, amp_pha = c[f"{name}.meta"]
    args = ao.Optics(amplitude_normalize=float(an), Holo_G_input="amp_pha" if amp_pha else "real_imag")
    out = at(ao.back_prop(c[f"{name}.holo"], c[f"{name}.d"], args), c[f"{name}.idx"])     # one row per channel
    ref = c[f"{name}.out"]
    if amp_pha:
        assert ao.rel_l2(out[0], ref[0]) < 2e-6
        assert ao.rel_l2(np.exp(1j * out[1]), np.exp(1j * ref[1].astype(np.float64))) < 5e-6
    else:
        assert ao.rel_l2(out, ref) < 2e-6


@pytest.mark.parametrize("pad", [False, True])
def test_adjoint_dot_product(pad):
    """<A x, y> = <x, A^H y> for the padded and unpadded operator (SURVEY.md section 4, item 4)."""
    rng = np.random.default_rng(7)
    B, N = 2, 32
    x = rng.standard_normal((B, 1, N, N)) + 1j * rng.standard_normal((B, 1, N, N))
    y = rng.standard_normal((B, 1, N, N)) + 1j * rng.standard_normal((B, 1, N, N))
    d = np.array([3e-4, 9e-4], dtype=np.float32)
    ax = ao.asm(x, 532e-9, d, 1.5e-6, pad)
    aty = ao.asm_adjoint(y, 532e-9, d, 1.5e-6, pad)
    lhs = np.vdot(y, ax)
    rhs = np.vdot(aty, x)
    assert abs(lhs - rhs) < 1e-10 * abs(lhs)


def test_unshifted_table_equals_centred_table():
    for n, pad in [(32, False), (32, True), (64, True)]:
        m = 2 * n if pad else n
        a = np.fft.ifftshift(ao.kz_centred(n, 532e-9, 0.2e-6, pad))
        b = ao.kz_unshifted(m, n, 532e-9, 0.2e-6)
        assert np.max(np.abs(a - b)) <= 1e-9 * np.max(a)
        assert (b == 0).mean() > 0.3      # evanescent clamp is exercised


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout only exists in the build container")
def test_live_reference_float64():
    """With complex128 input the reference runs in double end to end: the oracle must agree to ~1e-15,
    including the dtype-dependent rounding of the phase constant (fp32 d vs python float d)."""
    import torch
    ASM, Holo_Generator, Back_prop = ref_import.load()
    torch.manual_seed(3)
    B, N = 2, 32
    O = torch.randn(B, 1, N, N, dtype=torch.float64) + 1j * torch.randn(B, 1, N, N, dtype=torch.float64)
    for pad in (False, True):
        for d in (torch.tensor([[[[4e-4]]], [[[7e-3]]]]), 0.0031, torch.tensor(0.0031)):
            with torch.no_grad():
                r = ASM(O, 532e-9, d, 1.5e-6, zero_padding=pad).numpy()
            dn = d.numpy() if torch.is_tensor(d) else np.float64(d)
            assert ao.rel_l2(ao.asm(O.numpy(), 532e-9, dn, 1.5e-6, pad), r) < 1e-13


def test_unwrap_oracle_properties():
    """oracle/unwrap_oracle.py (Herraez 2002, the algorithm of skimage's 2-D unwrap_phase that utils/functions.py:44-59
    calls): residue-free surfaces are recovered exactly up to one global multiple of 2 pi, output - input is a multiple of
    2 pi, an unwrapped-range input is returned unchanged.  (Parity with scikit-image itself is unpinned: not installed.)"""
    from oracle import unwrap_oracle as uo
    rng = np.random.default_rng(11)
    y, x = np.mgrid[0:36, 0:28].astype(np.float64)
    true = 18 * np.exp(-((x - 13) ** 2 + (y - 20) ** 2) / (2 * 7.0 ** 2)) + 0.06 * x - 0.04 * y
    wrapped = np.angle(np.exp(1j * true)).astype(np.float32)
    got = uo.unwrap2d(wrapped)
    k = (got - wrapped) / (2 * np.pi)
    assert np.abs(k - np.round(k)).max() < 1e-5
    d = got - true
    assert np.abs(d - np.round(d.mean() / (2 * np.pi)) * 2 * np.pi).max() < 1e-4
    small = (0.5 * rng.random((1, 1, 16, 16))).astype(np.float32)      # MNIST-like phase in [0, 1): nothing to unwrap
    assert np.array_equal(uo.unwrap(small), small)


def test_oracle_matches_reference_any_size():
    """Sizes that are not powers of two (even padded / any unpadded): the oracle against the live reference's ASM and its
    autograd VJP (utils/Angular_Spectrum_Method.py:7-36).  Needs the checkout or the staged copy (baseline/_ref)."""
    import torch
    from oracle import ref_import
    if not ref_import.available():
        pytest.skip("reference not available")
    ASM = ref_import.load()[0]
    rng = np.random.default_rng(21)
    for n, pad in [(92, True), (92, False), (45, False), (30, True)]:
        O = (rng.standard_normal((2, 1, n, n)) + 1j * rng.standard_normal((2, 1, n, n))).astype(np.complex64)
        G = (rng.standard_normal((2, 1, n, n)) + 1j * rng.standard_normal((2, 1, n, n))).astype(np.complex64)
        d = np.array([0.7e-3, 1.3e-3], dtype=np.float32).reshape(2, 1, 1, 1)
        x = torch.from_numpy(O).clone().requires_grad_(True)
        U = ASM(x, 532e-9, torch.from_numpy(d), 1.5e-6, zero_padding=pad)
        gr = torch.autograd.grad(U, x, grad_outputs=torch.from_numpy(G).to(U.dtype))[0].numpy()
        assert ao.rel_l2(ao.asm(O, 532e-9, d, 1.5e-6, pad), U.detach().numpy()) < 2e-6, (n, pad)
        assert ao.rel_l2(ao.asm_adjoint(G, 532e-9, d, 1.5e-6, pad), gr) < 2e-6, (n, pad)
