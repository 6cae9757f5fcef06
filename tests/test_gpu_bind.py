"""Polynomial::bind on the device vs the oracle (mirrors dense.rs:613-625, 709-753, 1095-1118)."""
import numpy as np
import pytest

import jolt_b200
from jolt_b200 import HIGH_TO_LOW, LOW_TO_HIGH, Polynomial
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import CH_ONE, CH_ZERO, parity_table, rand_challenge, rand_full, rand_limbs, rand_limbs_full, wide_hi4

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sess():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.mark.parametrize("n", [1, 2, 5, 10, 11, 16])
@pytest.mark.parametrize("order", [HIGH_TO_LOW, LOW_TO_HIGH])
@pytest.mark.parametrize("kind", ["challenge125", "full254", "wide_hi4"])
def test_bind_matches_oracle(sess, n, order, kind):
    # a random half of the entries is drawn over the whole field (the top third included, which rand_limbs never
    # reaches); wide_hi4 takes the 4-row product with hi across the top limb's whole range
    t = rand_limbs(100 + n, 1 << n)
    full = np.random.Generator(np.random.PCG64(n)).integers(0, 2, size=1 << n).astype(bool)
    t[full] = rand_limbs_full(200 + n, 1 << n)[full]
    r = {"challenge125": rand_challenge(7 + n), "full254": rand_full(9 + n), "wide_hi4": wide_hi4(11 + n)}[kind]
    poly = Polynomial.new(sess, t)
    poly.bind_with_order(r, order)
    assert len(poly) == 1 << (n - 1)
    assert (poly.evals() == C.bind(t, r, order, threads=4)).all()
    poly.free()


@pytest.mark.parametrize("order", [HIGH_TO_LOW, LOW_TO_HIGH])
def test_full_bind_sequence_equals_evaluate(sess, order):
    # dense.rs:1095-1118: binding point[0..] HighToLow, or point[n-1..0] LowToHigh, yields evaluate(point)
    n = 10
    vals = O.random_fr(3, 1 << n)
    pt = O.random_fr(4, n)
    poly = Polynomial.from_ints(sess, vals)
    seq = pt if order == HIGH_TO_LOW else list(reversed(pt))
    for c in seq:
        poly.bind_with_order(c, order)
    assert poly.to_ints() == [O.evaluate(vals, pt)]


def test_bind_edge_values_and_special_challenges(sess):
    n = 8
    t = rand_limbs(1, 1 << n)
    t[:9] = C.ints_to_mont([0, 1, O.R_MOD - 1, 2, O.R_MOD - 2, 0, 0, 1, 1])
    for r_int in (0, 1, O.R_MOD - 1, 2):
        r = np.array(O.to_mont_limbs(r_int), dtype=np.uint64)
        for order in (HIGH_TO_LOW, LOW_TO_HIGH):
            poly = Polynomial.new(sess, t)
            poly.bind_with_order(r, order)
            assert (poly.evals() == C.bind(t, r, order)).all()
            poly.free()
    # parity tables (raw r - 1 at odd popcount, pairs (0, r - 1) / (r - 1, 0)) bound with 0 (the 4-row path) and 1
    # (the full product) select one side of every pair exactly: the result is a parity table again
    for inv in (False, True):
        t = parity_table(16, inv)
        for r in (CH_ZERO, CH_ONE):
            for order in (HIGH_TO_LOW, LOW_TO_HIGH):
                poly = Polynomial.new(sess, t)
                poly.bind_with_order(r, order)
                got = poly.evals()
                assert (got == C.bind(t, r, order, threads=4)).all()
                assert any((got == parity_table(15, i)).all() for i in (False, True))
                poly.free()


def test_bind_rejects_bad_input(sess):
    poly = Polynomial.new(sess, rand_limbs(1, 1))
    with pytest.raises(jolt_b200.JoltB200Error):       # "cannot bind a zero-variable polynomial"
        poly.bind(5)
    with pytest.raises(ValueError):                     # power-of-two assertion (dense_mlpoly.rs:28-32)
        Polynomial.new(sess, rand_limbs(1, 3))
    bad = np.array([2**64 - 1] * 4, dtype=np.uint64)    # non-canonical limbs
    p2 = Polynomial.new(sess, rand_limbs(1, 4))
    with pytest.raises(jolt_b200.JoltB200Error):
        p2.bind(bad)


@pytest.mark.parametrize("order", [HIGH_TO_LOW, LOW_TO_HIGH])
def test_bind_2pow22_round_matches_oracle(sess, order):
    # BASELINE config 2 size: one round at 2^22 against the (threaded) C oracle
    t = rand_limbs(0xB200, 1 << 22)
    r = rand_challenge(0xB201)
    poly = Polynomial.new(sess, t)
    poly.bind_with_order(r, order)
    assert (poly.evals() == C.bind(t, r, order, threads=C.max_threads())).all()
    poly.free()
