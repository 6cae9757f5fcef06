"""The operand families of tests/gpu_util.py produce canonical limbs in the range each one promises."""
import numpy as np
import pytest

from oracle import bn254 as O
from oracle import coracle as C
from jolt_b200 import HIGH_TO_LOW, LOW_TO_HIGH
from gpu_util import (CH_ONE, CH_ZERO, R_MINUS_1, const_table, limbs_below, limbs_of, parity_table, rand_limbs_full,
                      top_band, wide_hi4)


def raw_ints(a):
    return [sum(int(row[k]) << (64 * k) for k in range(4)) for row in np.asarray(a).reshape(-1, 4)]


@pytest.mark.parametrize("p", [O.R_MOD, O.Q_MOD])
def test_rand_limbs_full_covers_the_whole_field(p):
    a = rand_limbs_full(5, 1 << 14, p)
    assert a.dtype == np.uint64 and a.shape == (1 << 14, 4)
    v = raw_ints(a)
    assert max(v) < p and limbs_below(a, p).all()
    top = sum(x >> 253 != 0 for x in v) / len(v)     # [2^253, p) is about a third of the field
    assert abs(top - (p - (1 << 253)) / p) < 0.02
    assert (rand_limbs_full(5, 1 << 14, p) == a).all()    # seeded: the same draw every time


def test_top_band_is_just_below_r():
    a = top_band(7, 1 << 12)
    v = raw_ints(a)
    assert all(O.R_MOD - (1 << 128) <= x < O.R_MOD for x in v)
    assert len(set(v)) == len(v)
    assert min(v) < O.R_MOD - (1 << 127)               # the draw spans the band, not only its top


def test_limbs_below_compares_most_significant_first():
    r = O.R_MOD
    rows = np.stack([limbs_of(x) for x in (0, r - 1, r, r + 1, (1 << 256) - 1, r - (1 << 200))])
    assert limbs_below(rows, r).tolist() == [True, True, False, False, False, True]


@pytest.mark.parametrize("invert", [False, True])
def test_parity_table_and_its_binds(invert):
    n = 6
    t = parity_table(n, invert)
    for x in range(1 << n):
        odd = bin(x).count("1") % 2 == 1
        want = R_MINUS_1 if odd != invert else np.zeros(4, dtype=np.uint64)
        assert (t[x] == want).all()
    assert (parity_table(n, not invert) + t == R_MINUS_1).all()
    assert raw_ints(CH_ZERO) == [0] and C.mont_to_ints(CH_ONE) == [1]
    # challenges 0 and 1 keep a parity table (plain or inverted) in every round and both orders
    for order in (HIGH_TO_LOW, LOW_TO_HIGH):
        cur = t
        for rnd in range(n):
            k = n - rnd
            assert any((cur == parity_table(k, inv)).all() for inv in (False, True)), (order, rnd)
            cur = C.bind(cur, CH_ONE if (rnd * 5 + order) % 3 else CH_ZERO, order)


def test_const_tables():
    assert (const_table(3, 0) == 0).all()
    assert (const_table(3, O.R_MOD - 1) == R_MINUS_1).all() and const_table(3, 0).shape == (8, 4)


def test_wide_hi4_spans_the_top_limb():
    one = wide_hi4(3)
    assert one.shape == (4,) and one[0] == 0 and one[1] == 0
    a = wide_hi4(9, 1 << 12)
    assert (a[:, 0] == 0).all() and (a[:, 1] == 0).all()
    assert limbs_below(a, O.R_MOD).all()
    top = a[:, 3]
    assert (top >= np.uint64(1 << 61)).mean() > 0.25   # past the 61-bit mask of a 125-bit challenge
    assert (top < np.uint64(1 << 61)).mean() > 0.5
    assert (a[:, 2] >= np.uint64(1 << 63)).any()
