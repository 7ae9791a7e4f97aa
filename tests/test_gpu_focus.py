"""GPU: focal stacks (asm_b200_focal_stack) against the float64 oracle on every kernel family they touch, consistency
with the single-distance call, determinism, memory of a moments-only call, and autofocus."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import asm_oracle as ao

pytestmark = pytest.mark.gpu

ARGS = ao.Optics()
LAMB, PX = ARGS.wavelength, ARGS.pixel_size


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import style_transfer_based_holographic_imaging_b200 as p
    p._lib.load()
    return p


def _rel(a, b):
    return float(np.linalg.norm((a - b).ravel()) / np.linalg.norm(b.ravel()))


def _oracle_stack(field, z, pad):
    """field [B,N,N] complex128, z [B,K] -> oracle planes [B,K,N,N] complex128."""
    b, k = z.shape
    rep = np.repeat(field[:, None], k, axis=0)                      # [B*K,1,N,N], sample-major
    u = ao.asm(rep, LAMB, z.reshape(-1), PX, zero_padding=pad)
    return u.reshape(b, k, field.shape[-1], field.shape[-1])


def _moments64(u):
    a = np.abs(u).reshape(u.shape[0], u.shape[1], -1)
    return np.stack([a.sum(-1), (a ** 2).sum(-1), (a ** 4).sum(-1)], axis=-1)


def _const_amp_phase_stack(pkg, amp, phase, z, pad, out_mode, with_moments):
    """The C ABI with IN_CONST_AMP_PHASE (the loaders' constant amplitude): not exposed by focal_stack."""
    L = pkg._lib
    lib = L.load()
    b, n = phase.shape[0], phase.shape[-1]
    k = z.shape[1]
    zd = L.Z_F64 if z.dtype == torch.float64 else L.Z_F32
    ws = torch.empty(lib.asm_b200_focal_stack_workspace_bytes(b, k, n, int(pad)), dtype=torch.uint8, device=phase.device)
    out0 = torch.empty((b, k, n, n), dtype=torch.complex64, device=phase.device)
    mom = torch.empty((b, k, 3), dtype=torch.float64, device=phase.device) if with_moments else None
    p = lambda t: ctypes.c_void_p(0 if t is None else t.data_ptr())
    rc = lib.asm_b200_focal_stack(p(amp), p(phase), p(z), zd, k, p(out0), None, p(mom), b, n, int(pad),
                                  L.IN_CONST_AMP_PHASE, out_mode, LAMB, PX, 1.0, p(ws), ws.numel(),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    L.check(rc)
    return out0, mom


# (N, zero_padding, z dtype, input): every FFT family the stack runs (generic <= 512 and 4096, k32t at 1024, k64 at
# 2048, padded variants) and the matrix-product path (92 padded)
CASES = [
    (32, False, torch.float32, "complex"), (64, False, torch.float64, "complex"), (128, True, torch.float32, "complex"),
    (128, True, torch.float32, "hologram"), (128, True, torch.float64, "const_amp_phase"),
    (256, False, torch.float64, "complex"), (512, False, torch.float32, "complex"), (512, True, torch.float64, "complex"),
    (1024, False, torch.float32, "complex"), (1024, False, torch.float64, "hologram"),
    (1024, True, torch.float32, "complex"), (1024, True, torch.float32, "const_amp_phase"),
    (2048, False, torch.float64, "complex"), (2048, False, torch.float32, "const_amp_phase"),
    (4096, False, torch.float32, "complex"), (92, True, torch.float64, "complex"), (92, True, torch.float32, "hologram"),
]


@pytest.mark.parametrize("n,pad,zdtype,inp", CASES, ids=[f"{c[0]}{'p' if c[1] else ''}-{str(c[2])[-7:]}-{c[3]}" for c in CASES])
def test_parity_with_oracle(pkg, n, pad, zdtype, inp):
    rng = np.random.default_rng(n + 7 * pad)
    b, k = (1, 2) if n >= 2048 else (2, 3)
    dev = torch.device("cuda:0")
    z = (rng.uniform(-20e-3, 20e-3, (b, k))).astype(np.float32 if zdtype == torch.float32 else np.float64)
    z[0, 0] = 20e-3
    zt = torch.from_numpy(z).to(dev)
    if inp == "complex":
        x = (rng.standard_normal((b, n, n)) + 1j * rng.standard_normal((b, n, n))).astype(np.complex64)
        field = x.astype(np.complex128)
        xt, holo = torch.from_numpy(x).to(dev), False
    elif inp == "hologram":
        x = rng.uniform(0.0, 2.0, (b, n, n)).astype(np.float32)
        field = np.sqrt(x.astype(np.float64)).astype(np.complex128)
        xt, holo = torch.from_numpy(x).to(dev), True
    else:
        phase = rng.uniform(-np.pi, np.pi, (b, n, n)).astype(np.float32)
        field = ao.object_field(np.float32(0.6), phase, ARGS).astype(np.complex128)
    ref = _oracle_stack(field, z, pad)
    mref = _moments64(ref)
    outs = {}
    if inp == "const_amp_phase":
        amp = torch.tensor([0.6], dtype=torch.float32, device=dev)
        u, mom = _const_amp_phase_stack(pkg, amp, torch.from_numpy(phase).to(dev), zt, pad, pkg._lib.OUT_COMPLEX, True)
        outs["complex"] = u
        outs["moments"] = mom
    else:
        outs["complex"], outs["moments"] = pkg.focal_stack(xt, zt, LAMB, PX, pad, hologram=holo, output="complex", moments=True)
        outs["intensity"] = pkg.focal_stack(xt, zt, LAMB, PX, pad, hologram=holo, output="intensity")
        outs["abs_angle"] = pkg.focal_stack(xt, zt, LAMB, PX, pad, hologram=holo, output="abs_angle")
        outs["moments_only"] = pkg.focal_stack(xt, zt, LAMB, PX, pad, hologram=holo, output=None, moments=True)
    torch.cuda.synchronize()
    u = outs["complex"].cpu().numpy()
    for i in range(b):
        for j in range(k):
            assert _rel(u[i, j], ref[i, j]) < 1e-4, (i, j, _rel(u[i, j], ref[i, j]))
            if inp != "const_amp_phase":
                assert _rel(outs["intensity"][i, j].cpu().numpy(), np.abs(ref[i, j]) ** 2) < 1e-4
                a, ang = outs["abs_angle"][0][i, j].cpu().numpy(), outs["abs_angle"][1][i, j].cpu().numpy()
                assert _rel(a * np.exp(1j * ang), ref[i, j]) < 1e-4
    for key in ("moments", "moments_only"):
        if key in outs:
            m = outs[key].cpu().numpy()
            assert np.max(np.abs(m - mref) / mref) < 1e-5, (key, np.max(np.abs(m - mref) / mref))
    if "moments_only" in outs:
        assert torch.equal(outs["moments_only"], outs["moments"])


@pytest.mark.parametrize("n,pad", [(256, False), (128, True), (1024, False), (1024, True), (2048, False), (92, True)])
def test_single_plane_matches_forward(pkg, n, pad):
    rng = np.random.default_rng(1)
    dev = torch.device("cuda:0")
    x = torch.from_numpy((rng.standard_normal((2, 1, n, n)) + 1j * rng.standard_normal((2, 1, n, n))).astype(np.complex64)).to(dev)
    z = torch.tensor([[3e-3], [-1.2e-3]], dtype=torch.float32, device=dev)
    stack = pkg.focal_stack(x, z, LAMB, PX, pad, output="complex")
    one = pkg.asm_forward_raw(x, z.reshape(2, 1, 1, 1), LAMB, PX, pad)
    assert _rel(stack[:, 0].cpu().numpy(), one[:, 0].cpu().numpy()) <= 2e-6


@pytest.mark.parametrize("b,k,n,pad", [(3, 37, 256, False), (2, 9, 1024, False), (2, 7, 2048, False), (5, 11, 128, True)])
def test_many_chunks_and_groups(pkg, b, k, n, pad):
    """Per-sample [B,K] distances; B K planes spanning several chunks (small N) or plane groups (large N)."""
    rng = np.random.default_rng(2)
    dev = torch.device("cuda:0")
    x = torch.from_numpy((rng.standard_normal((b, n, n)) + 1j * rng.standard_normal((b, n, n))).astype(np.complex64)).to(dev)
    z = torch.from_numpy(rng.uniform(-5e-3, 5e-3, (b, k)).astype(np.float32)).to(dev)
    img, mom = pkg.focal_stack(x, z, LAMB, PX, pad, output="intensity", moments=True)
    rep = x.reshape(b, 1, 1, n, n).expand(b, k, 1, n, n).reshape(b * k, 1, n, n).contiguous()
    ref = pkg.asm_forward_raw(rep, z.reshape(-1, 1, 1, 1), LAMB, PX, pad).reshape(b, k, n, n)
    assert _rel(img.cpu().numpy(), (ref.abs() ** 2).cpu().numpy()) < 1e-5
    a = ref.abs().to(torch.float64).reshape(b, k, -1)
    mref = torch.stack([a.sum(-1), (a ** 2).sum(-1), (a ** 4).sum(-1)], -1)
    assert float(((mom - mref).abs() / mref).max()) < 1e-5


@pytest.mark.parametrize("n,pad", [(256, False), (1024, False), (2048, False), (92, True)])
def test_repeated_calls_bit_identical(pkg, n, pad):
    rng = np.random.default_rng(3)
    dev = torch.device("cuda:0")
    x = torch.from_numpy(rng.uniform(0, 1, (3, n, n)).astype(np.float32)).to(dev)
    z = [0.5e-3 * i for i in range(-3, 6)]
    runs = [pkg.focal_stack(x, z, LAMB, PX, pad, hologram=True, output="complex", moments=True) for _ in range(3)]
    runs.append((None, pkg.focal_stack(x, z, LAMB, PX, pad, hologram=True, output=None, moments=True)))
    for img, mom in runs[1:]:
        if img is not None:
            assert torch.equal(img, runs[0][0])
        assert torch.equal(mom, runs[0][1])


def test_moments_only_allocates_no_stack(pkg):
    b, k, n = 16, 16, 1024
    dev = torch.device("cuda:0")
    x = torch.rand(b, n, n, device=dev)
    z = torch.linspace(-4e-3, 4e-3, k, device=dev)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.max_memory_allocated(dev)
    mom = pkg.focal_stack(x, z, LAMB, PX, hologram=True, output=None, moments=True)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated(dev) - base < b * k * n * n * 4
    assert tuple(mom.shape) == (b, k, 3) and bool(torch.isfinite(mom).all())


def test_exact_refocus(pkg):
    """Back-propagating U = ASM(0.6 e^{i phi}, z0) by -z0 gives back a uniform amplitude: the pick is z0 exactly."""
    rng = np.random.default_rng(4)
    dev = torch.device("cuda:0")
    b, n = 4, 256
    grid = np.round(np.arange(0.2, 2.01, 0.1), 3) * 1e-3
    idx = np.array([3, 7, 12, 18])
    phi = rng.uniform(-np.pi, np.pi, (b, 1, n, n)).astype(np.float32)
    o = torch.from_numpy(0.6 * np.exp(1j * phi).astype(np.complex64)).to(dev)
    z0 = torch.from_numpy(grid[idx].reshape(b, 1, 1, 1)).to(dev)
    u = pkg.ASM(o, LAMB, z0, PX)
    for metric in ("tamura", "variance"):
        z_best, index, curve = pkg.autofocus(u.detach(), torch.from_numpy(-grid).to(dev), LAMB, PX, hologram=False,
                                             metric=metric, select="min")
        assert index.cpu().numpy().tolist() == idx.tolist()
        assert np.allclose(z_best.cpu().numpy(), -grid[idx], rtol=0, atol=0)
        assert tuple(curve.shape) == (b, len(grid))


def test_autofocus_mnist_holograms(pkg, mnist_golden):
    """The 100 bundled MNIST samples: Tamura minimum of the back-propagated amplitude over 0 .. 1.2 mm (25 candidates)
    lies within one step of the distance each hologram was generated at."""
    dev = torch.device("cuda:0")
    ph = mnist_golden["gt_phase"].reshape(100, 1, 128, 128)
    dc = mnist_golden["distance_content"].reshape(100)
    holo = ao.holo_generator(np.float32(0.6), ph, dc.reshape(100, 1, 1, 1), ARGS)
    zs = np.round(np.arange(0.0, 1.2 + 1e-9, 0.05), 3)
    z = torch.from_numpy(ao.metres(-zs, ARGS)).to(dev)
    h = torch.from_numpy(holo.astype(np.float32)).to(dev)
    z_best, index, curve = pkg.autofocus(h, z, LAMB, PX, hologram=True, metric="tamura", select="min")
    picked = zs[index.cpu().numpy()]
    err = np.abs(picked - dc)
    assert np.all(err <= 0.05 + 1e-6), (np.sum(err > 0.05 + 1e-6), err.max())
    assert tuple(curve.shape) == (100, 25)
