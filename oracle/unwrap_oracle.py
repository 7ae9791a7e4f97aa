"""TEST INFRASTRUCTURE (never imported by the product path): CPU restatement of 2-D phase unwrapping by reliability
sorting (Herraez, Burton, Lalor, Gdeisat, Appl. Opt. 41, 7437 (2002)) -- the algorithm behind
``skimage.restoration.unwrap_phase`` for 2-D input, which ``utils/functions.py:44-59`` of the reference calls per image.

PARITY UNPINNED against scikit-image itself: the package is not installed in this image, not vendored by the reference
(requirements.txt has no pin for it) and the reference ships no unwrapped golden vectors.  This file restates the published
steps; `tests/test_oracle.py` pins it through properties every correct unwrapper has (exact recovery of residue-free surfaces
up to one global multiple of 2 pi; output - input is an integer multiple of 2 pi), and `tests/test_gpu_unwrap.py` and
`tests/test_gpu_unwrap_exact.py` compare the CUDA kernel with it pixel for pixel.

Steps (numbered as in csrc/unwrap.cuh), one function each so that a test can replace exactly one of them:
  1. ``reliability``: wrapped second differences, borders a large constant;
  2. ``edges``: summed reliability of the two pixels of every edge, horizontal edges row by row, then vertical ones;
  3. ``order``: stable ascending sort of the edge keys;
  4. ``merge``: sequential group merging along the sorted edges, with the jump rule ``jump`` and the tie rule
     ``group2_joins`` (a single pixel joins its neighbour's group, else the smaller group joins the larger, ties: the first
     pixel's group joins); returns the integer 2 pi increment of every pixel;
  5. ``compose``: unwrapped = fl32(wrapped + 2 pi * increment), the sum in double.
The reliabilities, keys and jump comparisons are the kernel's fp32 operations in the kernel's order, and both sorts are
stable with the same tie order, so the increments are exact integers that the kernel must reproduce on every pixel.
"""
from __future__ import annotations

import numpy as np

PI = np.float32(np.pi)
TWO_PI = np.float32(2 * np.pi)
BORDER = np.float32(9999999.0)


def _wrap(x):
    x = x.astype(np.float32)
    return np.where(x > PI, x - TWO_PI, np.where(x < -PI, x + TWO_PI, x)).astype(np.float32)


def reliability(ph: np.ndarray) -> np.ndarray:
    """[H, W] fp32 wrapped phase -> [H, W] fp32 reliability (small = reliable)."""
    ph = ph.astype(np.float32)
    h, w = ph.shape
    rel = np.full((h, w), BORDER, dtype=np.float32)
    c = ph[1:-1, 1:-1]
    H = _wrap(ph[1:-1, :-2] - c) - _wrap(c - ph[1:-1, 2:])
    V = _wrap(ph[:-2, 1:-1] - c) - _wrap(c - ph[2:, 1:-1])
    D1 = _wrap(ph[:-2, :-2] - c) - _wrap(c - ph[2:, 2:])
    D2 = _wrap(ph[:-2, 2:] - c) - _wrap(c - ph[2:, :-2])
    rel[1:-1, 1:-1] = (H * H + V * V) + (D1 * D1 + D2 * D2)
    return rel


def edges(rel: np.ndarray):
    """[H, W] reliability -> (key fp32, p1, p2) per edge in the kernel's edge order: the H (W - 1) horizontal edges
    (i, j)-(i, j + 1) row by row, then the (H - 1) W vertical edges (i, j)-(i + 1, j).  p1, p2 are flat pixel indices."""
    h, w = rel.shape
    idx = np.arange(h * w).reshape(h, w)
    p1 = np.concatenate([idx[:, :-1].reshape(-1), idx[:-1, :].reshape(-1)])
    p2 = np.concatenate([idx[:, 1:].reshape(-1), idx[1:, :].reshape(-1)])
    flat = rel.reshape(-1)
    return (flat[p1] + flat[p2]).astype(np.float32), p1, p2


def order(key: np.ndarray) -> np.ndarray:
    """Visiting order of the edges: ascending key, ties in edge order (a stable sort, like cub's radix sort)."""
    return np.argsort(key, kind="stable")


def jump(d) -> int:
    """2 pi jump count of an edge from d = ph[p1] - ph[p2] (fp32)."""
    return -1 if d > PI else (1 if d < -PI else 0)


def group2_joins(size1: int, size2: int) -> bool:
    """Which group moves when the groups of p1 (size1 pixels) and p2 (size2) merge."""
    return True if size2 == 1 else (False if size1 == 1 else size1 > size2)


def merge(ph: np.ndarray, p1, p2, visit, jump=jump, group2_joins=group2_joins) -> np.ndarray:
    """Sequential merge along the edges in ``visit`` order -> int64 [H W] increments (a weighted union-find with
    per-node offsets and path halving, the same forest the kernel builds)."""
    flat = np.ascontiguousarray(ph, dtype=np.float32).reshape(-1)
    n = flat.size
    parent = list(range(n))
    off = [0] * n
    size = [1] * n

    def find(x):
        acc = 0
        while parent[x] != x:
            px = parent[x]
            if parent[px] != px:
                off[x] += off[px]
                parent[x] = parent[px]
            acc += off[x]
            x = parent[x]
        return x, acc

    fl = flat.tolist()
    p1l, p2l = p1.tolist(), p2.tolist()
    for k in visit.tolist():
        a, b = p1l[k], p2l[k]
        r1, o1 = find(a)
        r2, o2 = find(b)
        if r1 == r2:
            continue
        e = jump(np.float32(np.float32(fl[a]) - np.float32(fl[b])))
        if group2_joins(size[r1], size[r2]):        # every pixel of group 2 += o1 - e - o2
            off[r2] = o1 - e - o2
            parent[r2] = r1
            size[r1] += size[r2]
        else:                                       # every pixel of group 1 += o2 + e - o1
            off[r1] = o2 + e - o1
            parent[r1] = r2
            size[r2] += size[r1]
    return np.array([find(x)[1] for x in range(n)], dtype=np.int64)


def increments(ph: np.ndarray, reliability=reliability, edges=edges, order=order, merge=merge) -> np.ndarray:
    """One image [H, W] -> int64 [H, W] 2 pi increments.  Each keyword replaces one step (tests plant defects this way)."""
    ph = np.ascontiguousarray(ph, dtype=np.float32)
    key, p1, p2 = edges(reliability(ph))
    return merge(ph, p1, p2, order(key)).reshape(ph.shape)


def compose(ph: np.ndarray, inc: np.ndarray) -> np.ndarray:
    """fl32(ph + 2 pi k) with the sum in double: what the reference's float64 unwrap yields after its callers' .float()."""
    return (np.asarray(ph, dtype=np.float32).astype(np.float64) + 2 * np.pi * inc.astype(np.float64)).astype(np.float32)


def unwrap2d(ph: np.ndarray) -> np.ndarray:
    """One image [H, W] -> unwrapped float32 [H, W]."""
    ph = np.ascontiguousarray(ph, dtype=np.float32)
    return compose(ph, increments(ph))


def unwrap(x: np.ndarray) -> np.ndarray:
    """[B, 1, H, W] or [B, H, W] -> [B, 1, H, W] (the shape utils/functions.py:58 returns)."""
    x = np.asarray(x)
    imgs = x.reshape((-1,) + x.shape[-2:])
    return np.stack([unwrap2d(im) for im in imgs])[:, None]
