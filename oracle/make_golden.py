"""Generate tests/golden/* from the UNMODIFIED reference imported live (needs the reference checkout).

TEST INFRASTRUCTURE ONLY.  Run:  python oracle/make_golden.py
  * tests/golden/mnist_holo.npz   -- the reference's bundled fixtures (test_data/*.pt, 20 batches x 5 samples,
    N=128): gt_phase (stored losslessly as 8-bit codes, the phases are k/255), distance_content, distance_style and the
    stored hologram ``content_holo`` at MNIST_SAMPLES fixed positions per sample.  gt_amplitude is the constant 0.6
    (asserted here) and is not stored.
  * tests/golden/ref_cases.npz    -- outputs of the reference's ASM / Holo_Generator / Back_prop and the gradients
    PyTorch autograd derives from them, for the shapes/optics nothing in test_data pins (complex field, amp/phase,
    Back_prop, no-pad, evanescent optics, z up to 20 mm, negative z).  The inputs are not stored: ``ref_case_inputs``
    draws them again from one seeded torch CPU generator, and a CRC of each input checks that the draws still match.
  * tests/golden/ref_signatures.json -- the parameter names and defaults of the reference's three entry points.
Seeds and shapes are fixed, so the files are reproducible with the same torch build.
"""
from __future__ import annotations

import inspect
import json
import os
import sys
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_import  # noqa: E402
from oracle.asm_oracle import Optics  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
SEED = 20261018                  # torch CPU generator of every ref_cases input
SAMPLES = 512                    # stored positions per image-sized output of a ref case
MNIST_SAMPLES = 256              # stored positions per MNIST hologram
PHASE_LEVELS = (np.arange(256) / 255).astype(np.float32)    # every value the bundled MNIST phases take

ASM_CASES = [  # name, B, N, pad, lamb, px, zmax
    ("asm_n32", 3, 32, False, 532e-9, 1.5e-6, 1e-3),
    ("asm_n32_pad", 3, 32, True, 532e-9, 1.5e-6, 1e-3),
    ("asm_n64_far", 2, 64, False, 532e-9, 1.5e-6, 20e-3),
    ("asm_n64_pad_far", 2, 64, True, 532e-9, 1.5e-6, 20e-3),
    ("asm_n64_evan", 2, 64, False, 532e-9, 0.2e-6, 50e-6),       # 55 % of bins evanescent -> kz clamp
    ("asm_n32_pad_evan", 2, 32, True, 532e-9, 0.2e-6, 50e-6),
    ("asm_n128_neg", 1, 128, False, 633e-9, 2.0e-6, -6e-3),      # negative z (back-focus)
    ("asm_n128_pad", 1, 128, True, 532e-9, 1.5e-6, 0.8e-3),
]
HG_CASES = [  # name, B, N, optics kwargs, d range (normalised mm)
    ("hg_n32", 3, 32, dict(), (0.3, 0.9)),
    ("hg_n64_norm", 2, 64, dict(phase_normalize=2 * np.pi, distance_normalize=2.5, distance_normalize_constant=0.4), (-0.2, 0.6)),
    ("hg_n128_neg", 1, 128, dict(), (-0.8, -0.2)),
]
BP_CASES = [  # name, B, N, Holo_G_input, amplitude_normalize
    ("bp_n64_amp_pha", 2, 64, "amp_pha", 1.7), ("bp_n64_re_im", 2, 64, "real_imag", 0.5),
    ("bp_n32_amp_pha", 1, 32, "amp_pha", -1.0),
]
IMAGE_OUTPUTS = {"asm": ["U", "gO"], "hg": ["I", "amp", "ph", "U", "gA", "gP", "gA2", "gP2"], "bp": ["out"]}


def ref_case_inputs() -> dict:
    """Inputs and meta of every ref case, in the draw order the reference was run with."""
    g = torch.Generator().manual_seed(SEED)

    def rnd(*s):
        return torch.rand(*s, generator=g)

    def rndn(*s):
        return torch.randn(*s, generator=g)

    out = {}
    for name, B, N, pad, lamb, px, zmax in ASM_CASES:
        O = (rndn(B, 1, N, N) + 1j * rndn(B, 1, N, N)).to(torch.complex64)
        d = ((0.2 + 0.8 * rnd(B, 1, 1, 1)) * zmax).float()
        G = (rndn(B, 1, N, N) + 1j * rndn(B, 1, N, N)).to(torch.complex64)   # cotangent
        out.update({f"{name}.O": O.numpy(), f"{name}.d": d.numpy(), f"{name}.G": G.numpy(),
                    f"{name}.meta": np.array([B, N, int(pad), lamb, px], dtype=np.float64)})
    for name, B, N, kw, (dlo, dhi) in HG_CASES:
        args = Optics(**kw)
        A = (0.5 + 0.5 * rnd(B, 1, N, N)).float()
        P = rnd(B, 1, N, N).float() * (1.0 if kw else 2 * np.pi)
        d = (dlo + (dhi - dlo) * rnd(B, 1, 1, 1)).float()
        W = rndn(B, 1, N, N).float()
        Wa, Wp = rndn(B, 1, N, N).float(), rndn(B, 1, N, N).float()    # cotangents of the (abs, angle) outputs
        out.update({f"{name}.A": A.numpy(), f"{name}.P": P.numpy(), f"{name}.d": d.numpy(), f"{name}.W": W.numpy(),
                    f"{name}.Wa": Wa.numpy(), f"{name}.Wp": Wp.numpy(),
                    f"{name}.meta": np.array([B, N, args.wavelength, args.pixel_size, args.phase_normalize,
                                              args.distance_normalize, args.distance_normalize_constant])})
    for name, B, N, kind, an in BP_CASES:
        holo = (rnd(B, 1, N, N) * 1.5 + 0.05).float()
        d = (0.2 + 0.8 * rnd(B, 1, 1, 1)).float()
        out.update({f"{name}.holo": holo.numpy(), f"{name}.d": d.numpy(),
                    f"{name}.meta": np.array([B, N, an, 1.0 if kind == "amp_pha" else 0.0])})
    return out


def crc(a: np.ndarray) -> int:
    return zlib.crc32(np.ascontiguousarray(a).tobytes())


def at(x, idx) -> np.ndarray:
    """Values of an image-sized output at the stored positions ``idx`` (flat into [B,1,N,N]); a two-channel Back_prop
    output [B,2,N,N] gives one row per channel."""
    x = np.asarray(x)
    if x.shape[1] == 2:
        return np.stack([x[:, :1].reshape(-1)[idx], x[:, 1:].reshape(-1)[idx]])
    return x.reshape(-1)[idx]


def save_ref_cases(outputs: dict, path: str) -> None:
    """Store the reference's full ``outputs`` of every case as SAMPLES fixed positions per image-sized output
    (``name.idx``), per-sample scalars whole, the meta and a CRC of each input (``name.crc.<input>``)."""
    inputs = ref_case_inputs()
    rng = np.random.default_rng(SEED)
    keep = {}
    for family, cases in (("asm", ASM_CASES), ("hg", HG_CASES), ("bp", BP_CASES)):
        for case in cases:
            name, B, N = case[:3]
            idx = np.sort(rng.choice(B * N * N, min(SAMPLES, B * N * N), replace=False)).astype(np.int64)
            keep[f"{name}.idx"] = idx
            for k in IMAGE_OUTPUTS[family]:
                keep[f"{name}.{k}"] = at(outputs[f"{name}.{k}"], idx)
            for k in ("gd", "gd2"):
                if f"{name}.{k}" in outputs:
                    keep[f"{name}.{k}"] = outputs[f"{name}.{k}"]
            keep[f"{name}.meta"] = inputs[f"{name}.meta"]
            for k, v in inputs.items():
                if k.startswith(name + ".") and not k.endswith(".meta"):
                    keep[f"{name}.crc.{k[len(name) + 1:]}"] = np.int64(crc(v))
    np.savez_compressed(path, **keep)


def save_mnist(phase, holo, distance_content, distance_style, path: str) -> None:
    """phase, holo: [20,5,1,128,128] float32.  Phases go in as 8-bit codes (lossless, asserted), holograms as
    MNIST_SAMPLES fixed positions of each 128 x 128 image (``holo_idx``)."""
    codes = np.rint(phase * 255).astype(np.uint8)
    assert np.array_equal(PHASE_LEVELS[codes], phase), "gt_phase is expected to take the values k/255 only"
    n = holo.shape[-1] * holo.shape[-2]
    idx = np.sort(np.random.default_rng(SEED).choice(n, MNIST_SAMPLES, replace=False)).astype(np.int64)
    np.savez_compressed(path, gt_phase_code=codes, holo_idx=idx,
                        content_holo=holo.reshape(*holo.shape[:2], n)[..., idx].astype(np.float32),   # [20,5,K]
                        distance_content=distance_content.astype(np.float32),                          # [20,5,1,1,1]
                        distance_style=distance_style.astype(np.float32), amplitude=np.float32(0.6))


def mnist_fixtures():
    td = os.path.join(ref_import.CHECKOUT, "test_data")
    ld = lambda name, i: torch.load(os.path.join(td, f"test_{name}_{i}.pt"), map_location="cpu").numpy()
    phase, holo, dc, ds = [], [], [], []
    for i in range(20):
        amp = ld("gt_amplitude", i)
        assert np.all(amp == np.float32(0.6)), "gt_amplitude is expected to be the constant 0.6"
        phase.append(ld("gt_phase", i))
        holo.append(ld("content_holo", i))
        dc.append(ld("distance_content", i))
        ds.append(ld("distance_style", i))
    save_mnist(np.stack(phase).astype(np.float32), np.stack(holo).astype(np.float32), np.stack(dc), np.stack(ds),
               os.path.join(OUT, "mnist_holo.npz"))


def ref_cases():
    ASM, Holo_Generator, Back_prop = ref_import.load()
    inputs = ref_case_inputs()
    out = {}
    t = lambda k: torch.from_numpy(inputs[k])     # noqa: E731

    # ---- ASM, complex field in/out (utils/Angular_Spectrum_Method.py:7) ----
    for name, B, N, pad, lamb, px, zmax in ASM_CASES:
        Oq, dq, G = t(f"{name}.O").clone().requires_grad_(True), t(f"{name}.d").clone().requires_grad_(True), t(f"{name}.G")
        U = ASM(Oq, lamb, dq, px, zero_padding=pad)
        # the real scalar L = Re sum(conj(G) * U): what autograd gives for it is what a drop-in backward must reproduce
        L = torch.real(torch.sum(torch.conj(G.to(U.dtype)) * U))
        gO, gd = torch.autograd.grad(L, [Oq, dq])
        out.update({f"{name}.U": U.detach().numpy().astype(np.complex64), f"{name}.gO": gO.numpy(),
                    f"{name}.gd": gd.numpy()})

    # ---- Holo_Generator (utils/Forward_model.py:16-39) ----
    for name, B, N, kw, _ in HG_CASES:
        hg = Holo_Generator(Optics(**kw))
        A, P, d, W = t(f"{name}.A"), t(f"{name}.P"), t(f"{name}.d"), t(f"{name}.W")
        Aq, Pq, dq = A.clone().requires_grad_(True), P.clone().requires_grad_(True), d.clone().requires_grad_(True)
        I = hg(Aq, Pq, dq)
        gA, gP, gd = torch.autograd.grad(torch.sum(W * I), [Aq, Pq, dq])
        with torch.no_grad():
            amp, ph = hg(A, P, d, return_field=True)
            Uc = hg(A, P, d, complex_number=True)
        # gradients through the (abs, angle) outputs as well
        a2, p2 = hg(Aq, Pq, dq, return_field=True)
        gA2, gP2, gd2 = torch.autograd.grad(torch.sum(t(f"{name}.Wa") * a2) + torch.sum(t(f"{name}.Wp") * p2), [Aq, Pq, dq])
        out.update({f"{name}.I": I.detach().numpy(), f"{name}.amp": amp.numpy(), f"{name}.ph": ph.numpy(),
                    f"{name}.U": Uc.numpy().astype(np.complex64), f"{name}.gA": gA.numpy(), f"{name}.gP": gP.numpy(),
                    f"{name}.gd": gd.numpy(), f"{name}.gA2": gA2.numpy(), f"{name}.gP2": gP2.numpy(),
                    f"{name}.gd2": gd2.numpy()})

    # ---- Back_prop (utils/Forward_model.py:52-65) ----
    for name, B, N, kind, an in BP_CASES:
        bp = Back_prop(Optics(amplitude_normalize=an, Holo_G_input=kind))
        with torch.no_grad():
            r = bp(t(f"{name}.holo"), t(f"{name}.d"))
        out[f"{name}.out"] = r.numpy().astype(np.float32)

    save_ref_cases(out, os.path.join(OUT, "ref_cases.npz"))


def signatures():
    ASM, Holo_Generator, Back_prop = ref_import.load()
    rec = {}
    for key, fn in (("ASM", ASM), ("Holo_Generator.forward", Holo_Generator.forward), ("Back_prop.forward", Back_prop.forward)):
        ps = inspect.signature(fn).parameters.values()
        rec[key] = {"names": [p.name for p in ps],
                    "defaults": {p.name: p.default for p in ps if p.default is not inspect.Parameter.empty}}
    with open(os.path.join(OUT, "ref_signatures.json"), "w") as f:
        json.dump(rec, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    if not ref_import.available():
        sys.exit("reference checkout not present; golden vectors are generated from the reference only")
    os.makedirs(OUT, exist_ok=True)
    mnist_fixtures()
    ref_cases()
    signatures()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
