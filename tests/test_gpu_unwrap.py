"""Device-side phase unwrapping (asm_b200_unwrap, SURVEY.md 8f row 4) against the CPU restatement of the same algorithm
(oracle/unwrap_oracle.py) and against the properties any correct unwrapper has."""
import numpy as np
import pytest
import torch

from oracle import asm_oracle as ao
from oracle import unwrap_oracle as uo

pytestmark = pytest.mark.gpu


def _surface(rng, b, h, w, amp):
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    out = []
    for _ in range(b):
        cx, cy, s = rng.uniform(0.3, 0.7) * w, rng.uniform(0.3, 0.7) * h, rng.uniform(0.15, 0.3) * w
        tilt = rng.uniform(-0.1, 0.1, size=2)
        out.append(amp * np.exp(-((x - cx) ** 2 + (y - cy) ** 2) / (2 * s * s)) + tilt[0] * x + tilt[1] * y)
    return np.stack(out)[:, None]


def test_unwrap_recovers_smooth_surfaces_and_matches_oracle():
    import style_transfer_based_holographic_imaging_b200 as pkg
    rng = np.random.default_rng(5)
    for (b, h, w, amp) in [(3, 32, 32, 12.0), (2, 64, 48, 25.0), (5, 128, 128, 40.0)]:
        true = _surface(rng, b, h, w, amp)
        wrapped = np.angle(np.exp(1j * true)).astype(np.float32)
        got = pkg.unwrap(torch.from_numpy(wrapped).cuda()).cpu().numpy()
        assert got.shape == (b, 1, h, w) and got.dtype == np.float32
        k = (got - wrapped) / (2 * np.pi)
        assert np.abs(k - np.round(k)).max() < 1e-4                   # output - input is a multiple of 2 pi
        d = got - true                                                # residue-free: exact up to ONE global multiple of 2 pi
        for i in range(b):
            shift = np.round(d[i].mean() / (2 * np.pi)) * 2 * np.pi
            assert np.abs(d[i] - shift).max() < 1e-3, (b, h, w, i)
        if h * w <= 64 * 64:                                          # the sequential oracle is a pure-Python loop
            assert np.array_equal(got.view(np.int32), uo.unwrap(wrapped).view(np.int32))   # bit for bit


def test_unwrap_noisy_phase_matches_oracle_exactly():
    """With residues the result depends on the merge order.  The kernel computes the same fp32 keys as the oracle and both
    sort stably with the same tie order, so every increment agrees, and so does every value bit for bit."""
    import style_transfer_based_holographic_imaging_b200 as pkg
    rng = np.random.default_rng(6)
    true = _surface(rng, 2, 48, 48, 15.0) + 0.4 * rng.standard_normal((2, 1, 48, 48))
    wrapped = np.angle(np.exp(1j * true)).astype(np.float32)
    got = pkg.unwrap(torch.from_numpy(wrapped).cuda()).cpu().numpy()
    ref = uo.unwrap(wrapped)
    kg, kr = np.round((got - wrapped) / (2 * np.pi)), np.round((ref - wrapped) / (2 * np.pi))
    assert np.abs((got - wrapped) / (2 * np.pi) - kg).max() < 1e-4
    assert np.array_equal(kg, kr)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32))


def test_holo_generator_unwrap_on_device():
    """Holo_Generator(..., return_field=True, unwrap=True): the back-focus call of test_field_retrieval_mnist.py:126."""
    import style_transfer_based_holographic_imaging_b200 as pkg
    rng = np.random.default_rng(7)
    b, n = 3, 128
    amp = np.full((b, 1, n, n), 0.6, dtype=np.float32)
    ph = np.zeros((b, 1, n, n), dtype=np.float32)
    ph[:, :, 40:90, 40:90] = rng.random((b, 1, 50, 50)).astype(np.float32)
    d = np.full((b, 1, 1, 1), -0.2, dtype=np.float32)
    args = ao.Optics()
    hg = pkg.Holo_Generator(args).cuda()
    with torch.no_grad():
        a0, p0 = hg(torch.from_numpy(amp).cuda(), torch.from_numpy(ph).cuda(), torch.from_numpy(d).cuda(), return_field=True)
        a1, p1 = hg(torch.from_numpy(amp).cuda(), torch.from_numpy(ph).cuda(), torch.from_numpy(d).cuda(), return_field=True,
                    unwrap=True)
    assert p1.is_cuda and p1.shape == p0.shape and torch.equal(a0, a1)
    k = ((p1 - p0) / (2 * np.pi)).cpu().numpy()
    assert np.abs(k - np.round(k)).max() < 1e-4
