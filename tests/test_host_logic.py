"""CPU: host-side logic of the drop-in interface (no CUDA): signatures mirror the reference, distance handling,
no CPU fallback, shard arithmetic, and the CPU baseline port agrees with the oracle."""
import inspect
import json
import os

import numpy as np
import pytest
import torch

import style_transfer_based_holographic_imaging_b200 as pkg
from style_transfer_based_holographic_imaging_b200 import _lib as L
from style_transfer_based_holographic_imaging_b200 import functional as F_
from style_transfer_based_holographic_imaging_b200 import parallel
from oracle import asm_oracle as ao
from oracle import torch_port


def test_signatures_match_reference_names():
    sig = inspect.signature(pkg.ASM)
    assert list(sig.parameters)[:6] == ["O", "lamb", "d", "px", "requires_grad", "zero_padding"]
    assert sig.parameters["requires_grad"].default is True and sig.parameters["zero_padding"].default is False
    sig = inspect.signature(pkg.Holo_Generator.forward)
    assert list(sig.parameters) == ["self", "amplitude", "phase", "d", "return_field", "complex_number", "unwrap"]
    assert list(inspect.signature(pkg.Back_prop.forward).parameters) == ["self", "holo", "d"]
    # the package also mirrors the reference's module layout
    from style_transfer_based_holographic_imaging_b200.utils.Forward_model import Holo_Generator, Back_prop  # noqa
    from style_transfer_based_holographic_imaging_b200.utils.Angular_Spectrum_Method import ASM  # noqa


def test_signatures_equal_the_live_reference():
    """Parameter names and defaults against the reference's, as oracle/make_golden.py records them from its source
    (tests/golden/ref_signatures.json); ASM may take extra trailing parameters."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_signatures.json")) as f:
        ref = json.load(f)
    for key, fn in (("ASM", pkg.ASM), ("Holo_Generator.forward", pkg.Holo_Generator.forward),
                    ("Back_prop.forward", pkg.Back_prop.forward)):
        ps = inspect.signature(fn).parameters
        names = list(ps)[:len(ref[key]["names"])] if key == "ASM" else list(ps)
        assert names == ref[key]["names"], key
        assert {k: ps[k].default for k in ref[key]["defaults"]} == ref[key]["defaults"], key


def test_modules_take_any_args_object_and_have_no_parameters():
    hg = pkg.Holo_Generator(ao.Optics(phase_normalize=2.0))
    bp = pkg.Back_prop(ao.Optics(amplitude_normalize=1.5, Holo_G_input="real_imag"))
    assert list(hg.parameters()) == [] and list(bp.parameters()) == []
    assert hg.to("cpu") is hg and hg.phase_normalize == 2.0 and bp.input_type == "real_imag"


def test_no_cpu_fallback():
    x = torch.zeros(1, 1, 64, 64, dtype=torch.complex64)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.ASM(x, 532e-9, torch.tensor([[[[1e-3]]]]), 1.5e-6)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.Holo_Generator(ao.Optics())(torch.ones(1, 1, 64, 64), torch.zeros(1, 1, 64, 64), torch.ones(1, 1, 1, 1))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.Back_prop(ao.Optics())(torch.ones(1, 1, 64, 64), torch.ones(1, 1, 1, 1))


def test_prepare_distance_dtype_rules():
    dev = torch.device("cpu")
    z, zd = F_.prepare_distance(torch.full((3, 1, 1, 1), 2e-3), 3, dev)
    assert zd == L.Z_F32 and z.dtype == torch.float32 and z.shape == (3,)
    z, zd = F_.prepare_distance(2e-3, 3, dev)
    assert zd == L.Z_F64 and z.dtype == torch.float64 and z.shape == (3,)
    z, zd = F_.prepare_distance(torch.tensor(2e-3), 4, dev)
    assert zd == L.Z_F32 and z.shape == (4,)
    z, zd = F_.prepare_distance(torch.tensor(2e-3, dtype=torch.float64), 4, dev)
    assert zd == L.Z_F64 and z.shape == (4,)
    z, zd = F_.prepare_distance(torch.full((3, 1, 1, 1), 2e-3, dtype=torch.float16), 3, dev)
    assert zd == L.Z_F32 and z.dtype == torch.float32
    with pytest.raises(RuntimeError):
        F_.prepare_distance(torch.zeros(5), 3, dev)
    with pytest.raises(RuntimeError):
        F_.prepare_distance(torch.zeros(3, 2), 3, dev)


def test_shard_bounds_cover_the_batch_exactly():
    for batch in [0, 1, 5, 64, 512, 513]:
        for world in [1, 2, 3, 4, 8]:
            spans = [parallel.shard_bounds(batch, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == batch
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def test_cpu_baseline_port_agrees_with_oracle():
    """bench.py times oracle/torch_port.py as the CPU baseline; it must compute the same thing."""
    torch.manual_seed(0)
    O = torch.randn(2, 1, 64, 64, dtype=torch.complex64)
    d = torch.tensor([3e-4, 8e-3]).reshape(2, 1, 1, 1)
    for pad in (False, True):
        assert ao.rel_l2(torch_port.asm_cpu(O, 532e-9, d, 1.5e-6, pad).numpy(), ao.asm(O.numpy(), 532e-9, d.numpy(), 1.5e-6, pad)) < 2e-6
    assert ao.rel_l2(torch_port.adjoint_cpu(O, 532e-9, d, 1.5e-6).numpy(), ao.asm_adjoint(O.numpy(), 532e-9, d.numpy(), 1.5e-6)) < 2e-6
    i = torch_port.forward_intensity_cpu(O, 532e-9, d, 1.5e-6)
    assert i.dtype == torch.float32
    assert ao.rel_l2(i.numpy(), np.abs(ao.asm(O.numpy(), 532e-9, d.numpy(), 1.5e-6)) ** 2) < 2e-6
