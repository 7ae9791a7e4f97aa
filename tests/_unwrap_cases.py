"""Seeded wrapped-phase images shared by the unwrap oracle power test (CPU) and the exact GPU parity test.

Each generator maps (rng, h, w) to a float32 [h, w] image and works down to 3 x 3.  Together they reach the inputs where an
unwrapper goes wrong without a smooth test surface noticing: residues, exact key ties (quantised phases, the half-pi lattice,
a constant image), differences of exactly fl32(pi), a jump on every edge, and values outside [-pi, pi].
"""
from __future__ import annotations

import numpy as np

PI32 = np.float32(np.pi)


def _bump(rng, h, w):
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    cx, cy = rng.uniform(0.3, 0.7) * w, rng.uniform(0.3, 0.7) * h
    s = rng.uniform(0.15, 0.3) * max(h, w)
    amp = rng.uniform(8.0, 20.0)
    tilt = rng.uniform(-0.15, 0.15, size=2)
    return amp * np.exp(-((x - cx) ** 2 + (y - cy) ** 2) / (2 * s * s)) + tilt[0] * x + tilt[1] * y


def _wrap(t):
    return np.angle(np.exp(1j * t)).astype(np.float32)


def smooth(rng, h, w):
    """Residue-free surface: every correct unwrapper recovers it up to one global multiple of 2 pi."""
    return _wrap(_bump(rng, h, w))


def noisy(rng, h, w):
    """Surface plus noise: residues, so the result depends on the merge order."""
    return _wrap(_bump(rng, h, w) + 0.7 * rng.standard_normal((h, w)))


def quantised(rng, h, w):
    """8-bit codes k in 0..254 as 2 pi k / 255 - pi (the loaders' phases are k / 255): many equal differences, so equal
    reliabilities and edge keys."""
    t = (_bump(rng, h, w) + 0.3 * rng.standard_normal((h, w))) / (2 * np.pi)
    k = np.floor((t - np.floor(t)) * 255).astype(np.int64)
    return (np.float32(2 * np.pi / 255) * k.astype(np.float32) - PI32).astype(np.float32)


def half_pi(rng, h, w):
    """Phases in {-pi/2, 0, pi/2, pi} (fp32): differences of exactly fl32(pi), where > pi and >= pi part, and massive key
    ties."""
    return (np.float32(np.pi / 2) * (rng.integers(0, 4, size=(h, w)) - 1).astype(np.float32)).astype(np.float32)


def constant(rng, h, w):
    """One value everywhere: every interior reliability is 0, so every interior edge key ties."""
    return np.full((h, w), np.float32(rng.uniform(-np.pi, np.pi)), dtype=np.float32)


def steep_ramp(rng, h, w):
    """Unwrapped plane with slopes between pi and 2 pi per pixel: every edge carries a 2 pi jump."""
    sx, sy = rng.uniform(1.1 * np.pi, 1.9 * np.pi, size=2) * rng.choice([-1.0, 1.0], size=2)
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    return (sx * (x - w / 2) + sy * (y - h / 2)).astype(np.float32)


def out_of_range(rng, h, w):
    """A noisy wrapped surface with random pixels moved by +-2 pi: values up to +-3 pi, beyond what one wrap folds back."""
    return (noisy(rng, h, w) + np.float32(2 * np.pi) * rng.integers(-1, 2, size=(h, w)).astype(np.float32)).astype(np.float32)


def uniform(rng, h, w):
    """Independent uniform phases in [-pi, pi)."""
    return rng.uniform(-np.pi, np.pi, size=(h, w)).astype(np.float32)


GENERATORS = {"smooth": smooth, "noisy": noisy, "quantised": quantised, "half_pi": half_pi, "constant": constant,
              "steep_ramp": steep_ramp, "out_of_range": out_of_range}
NAMES = list(GENERATORS)


def case(name: str, h: int, w: int, seed: int = 0) -> np.ndarray:
    """One image of the named case, drawn from a seed fixed by (name, h, w, seed)."""
    rng = np.random.default_rng([NAMES.index(name), h, w, seed])
    return GENERATORS[name](rng, h, w)


def batch(h: int, w: int) -> np.ndarray:
    """[len(NAMES), h, w]: one image of every case."""
    return np.stack([case(n, h, w) for n in NAMES])


def tiny(seed: int, kind: str) -> np.ndarray:
    """A 3..8 x 3..8 image of independent uniform or half-pi lattice phases, shape and values drawn from ``seed``."""
    rng = np.random.default_rng(seed)
    h, w = (int(v) for v in rng.integers(3, 9, size=2))
    return {"uniform": uniform, "half_pi": half_pi}[kind](rng, h, w)


# Tiny images on which a merge tie rule alone decides increments.  Found by drawing seeds 0..399 of ``tiny`` and keeping
# the first whose increments change when that rule is altered:
#   equal_sizes: equal-size groups, the second pixel's group joins instead of the first's -> seed 13 (8 x 8, uniform);
#   single_pixel: without "a single pixel joins its neighbour's group"                    -> seed 3 (7 x 3, half-pi).
TINY = {"equal_sizes": (13, "uniform"), "single_pixel": (3, "half_pi")}
