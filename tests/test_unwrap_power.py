"""CPU: the unwrap oracle split into steps (oracle/unwrap_oracle.py) computes what the monolithic oracle it replaced
computed, and the shared cases (tests/_unwrap_cases.py) can see a wrong unwrapper.  Each planted defect swaps exactly one
step for a re-implementation of it; the same re-implementation without the defect must reproduce the increments exactly,
and with the defect it must change at least one increment of the case set.  The GPU parity tests compare the kernel on
these cases increment for increment, so each defect below is one the kernel cannot have without failing them."""
import numpy as np
import pytest

from oracle import unwrap_oracle as uo
import _unwrap_cases as uc

SHAPES = [(48, 48), (3, 3), (3, 40), (40, 3), (20, 24)]


def _case_set():
    imgs = [uc.case(n, h, w) for (h, w) in SHAPES for n in uc.NAMES]
    return imgs + [uc.tiny(seed, kind) for (seed, kind) in uc.TINY.values()]


CASES = _case_set()
REF = [uo.increments(ph) for ph in CASES]


def _unwrap2d_monolithic(ph):
    """The oracle before it was split into steps, kept verbatim apart from the return value (its fp32 composition
    ``flat + TWO_PI * inc`` is replaced by the increments themselves)."""
    ph = np.ascontiguousarray(ph, dtype=np.float32)
    h, w = ph.shape
    rel = uo.reliability(ph).reshape(-1)
    flat = ph.reshape(-1)
    idx = np.arange(h * w).reshape(h, w)
    p1 = np.concatenate([idx[:, :-1].reshape(-1), idx[:-1, :].reshape(-1)])
    p2 = np.concatenate([idx[:, 1:].reshape(-1), idx[1:, :].reshape(-1)])
    key = (rel[p1] + rel[p2]).astype(np.float32)
    order = np.argsort(key, kind="stable")
    parent = np.arange(h * w)
    off = np.zeros(h * w, dtype=np.int64)
    size = np.ones(h * w, dtype=np.int64)
    base = np.zeros(h * w, dtype=np.int64)

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

    for k in order:
        a, b = int(p1[k]), int(p2[k])
        r1, o1 = find(a)
        r2, o2 = find(b)
        if r1 == r2:
            continue
        d = np.float32(flat[a] - flat[b])
        e = -1 if d > uo.PI else (1 if d < -uo.PI else 0)
        inc1, inc2 = base[r1] + o1, base[r2] + o2
        group2_joins = True if size[r2] == 1 else (False if size[r1] == 1 else bool(size[r1] > size[r2]))
        if group2_joins:
            off[r2] = base[r2] + (inc1 - e - inc2) - base[r1]
            parent[r2] = r1
            size[r1] += size[r2]
        else:
            off[r1] = base[r1] + (inc2 + e - inc1) - base[r2]
            parent[r1] = r2
            size[r2] += size[r1]
    inc = np.zeros(h * w, dtype=np.int64)
    for x in range(h * w):
        r, o = find(x)
        inc[x] = base[r] + o
    return inc.reshape(h, w)


# ---- re-implemented steps: planted=False is the correct step, planted=True the defect ----------------------------------

def _reliability(planted):
    def step(ph):
        rel = uo.reliability(ph)
        if planted:                                   # border reliability 0 instead of the large constant
            rel[0, :] = rel[-1, :] = rel[:, 0] = rel[:, -1] = 0
        return rel
    return step


def _edges(planted):
    def step(rel):
        key, p1, p2 = uo.edges(rel)
        if planted:                                   # vertical edges ordered before horizontal ones
            h, w = rel.shape
            perm = np.roll(np.arange(key.size), -h * (w - 1))
            key, p1, p2 = key[perm], p1[perm], p2[perm]
        return key, p1, p2
    return step


def _order(planted):
    def step(key):                                    # ties in reverse edge order: what an unstable sort may do
        i = np.arange(key.size)
        return np.lexsort((-i if planted else i, key))
    return step


def _merge(jump=uo.jump, group2_joins=uo.group2_joins):
    return lambda ph, p1, p2, visit: uo.merge(ph, p1, p2, visit, jump=jump, group2_joins=group2_joins)


def _jump_at_pi(d):                                   # |d| >= pi counted as a jump
    return -1 if d >= uo.PI else (1 if d <= -uo.PI else 0)


def _equal_sizes_other_group(s1, s2):                 # equal-size groups: the second pixel's group joins
    return True if s2 == 1 else (False if s1 == 1 else s1 >= s2)


def _no_single_pixel_rule(s1, s2):                    # the smaller group joins, single pixels get no precedence
    return s1 > s2


PLANTS = {
    "border_reliability_zero": (dict(reliability=_reliability(False)), dict(reliability=_reliability(True))),
    "vertical_edges_first": (dict(edges=_edges(False)), dict(edges=_edges(True))),
    "unstable_sort": (dict(order=_order(False)), dict(order=_order(True))),
    "jump_at_pi_inclusive": (dict(merge=_merge()), dict(merge=_merge(jump=_jump_at_pi))),
    "equal_sizes_other_group_joins": (dict(merge=_merge()), dict(merge=_merge(group2_joins=_equal_sizes_other_group))),
    "no_single_pixel_rule": (dict(merge=_merge()), dict(merge=_merge(group2_joins=_no_single_pixel_rule))),
}


def test_split_oracle_matches_monolithic_oracle():
    for ph, k in zip(CASES, REF):
        assert np.array_equal(k, _unwrap2d_monolithic(ph)), ph.shape


def test_increments_are_the_unwrap_minus_input():
    for ph, k in zip(CASES, REF):
        got = uo.unwrap2d(ph).astype(np.float64)
        assert np.array_equal(np.round((got - ph.astype(np.float64)) / (2 * np.pi)).astype(np.int64), k), ph.shape


@pytest.mark.parametrize("name", list(PLANTS))
def test_planted_defect_changes_an_increment(name):
    correct, planted = PLANTS[name]
    for ph, k in zip(CASES, REF):
        assert np.array_equal(uo.increments(ph, **correct), k), (name, ph.shape)
    changed = sum(int((uo.increments(ph, **planted) != k).sum()) for ph, k in zip(CASES, REF))
    assert changed > 0, f"{name}: the case set cannot tell this defect from the oracle"


def test_tiny_cases_need_the_tie_rules():
    """Each searched tiny image changes its increments when the tie rule it was found for is altered."""
    for name, rule in [("equal_sizes", _equal_sizes_other_group), ("single_pixel", _no_single_pixel_rule)]:
        ph = uc.tiny(*uc.TINY[name])
        assert not np.array_equal(uo.increments(ph, merge=_merge(group2_joins=rule)), uo.increments(ph)), name


def test_value_composition_is_visible_bit_for_bit():
    """The oracle's value fl32(ph + 2 pi k), summed in double, differs from both fp32 compositions somewhere on the case
    set: the fp32 product then sum (two roundings) and a fused multiply-add with fl32(2 pi) (one rounding).  So comparing
    values bit for bit checks the composition as well as the increments."""
    two_rounding = fused = 0
    for ph, k in zip(CASES, REF):
        want = uo.compose(ph, k)
        two_rounding += int((want != (ph + uo.TWO_PI * k.astype(np.float32)).astype(np.float32)).sum())
        fused += int((want != (ph.astype(np.float64) + np.float64(uo.TWO_PI) * k).astype(np.float32)).sum())
    assert two_rounding > 0 and fused > 0, (two_rounding, fused)
