"""EqPolynomial::evals on the device vs the oracle (mirrors eq.rs:496-756, 238-263)."""
import numpy as np
import pytest

import jolt_b200
from jolt_b200 import EqPolynomial
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import rand_limbs, rand_limbs_full, wide_hi4

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sess():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.mark.parametrize("n", [0, 1, 2, 3, 5, 8, 11, 12, 13, 17])
@pytest.mark.parametrize("scaled", [False, True])
def test_eq_matches_oracle(sess, n, scaled):
    r = rand_limbs(300 + n, n)
    sc = rand_limbs(77, 1)[0] if scaled else None
    got = EqPolynomial.evals(sess, r, sc).evals()
    want = C.eq_evals(r, sc, threads=4 if n > 12 else 1)
    assert got.shape == want.shape and (got == want).all()


def test_eq_sums_to_one_and_pointwise(sess):
    n = 12
    r_int = O.random_fr(9, n)
    tab = EqPolynomial.evals(sess, C.ints_to_mont(r_int)).to_ints()
    assert sum(tab) % O.R_MOD == 1
    for x in (0, 1, 1234, (1 << n) - 1):
        v = 1
        for i in range(n):
            bit = (x >> (n - 1 - i)) & 1          # r[0] <-> MSB
            v = v * (r_int[i] if bit else 1 - r_int[i]) % O.R_MOD
        assert tab[x] == v


def test_eq_aligned_block_is_slice(sess):
    n = 14
    r = rand_limbs(5, n)
    full = EqPolynomial.evals(sess, r).evals()
    for start, size in ((0, 1 << 11), (3 << 11, 1 << 11), (3 << 12, 1 << 12), (1 << 13, 1 << 13), (0, 1 << 14), (7, 1)):
        got = EqPolynomial.evals_for_aligned_block(sess, r, start, size).evals()
        assert (got == full[start:start + size]).all()


@pytest.mark.parametrize("pattern,n", [("cycle", 3), ("cycle", 12), ("cycle", 17), ("stage_zero", 12), ("stage_zero", 13),
                                       ("stage_zero", 17)])
def test_eq_edge_coordinates_and_scales(sess, pattern, n):
    """Coordinates 0 (all-zero limbs: the 4-row product), 1 and r - 1 in turn; "stage_zero" makes the three
    register-stage variables of the streaming kernel (r[n - 11 .. n - 8)) zero, so it takes its hi4 path with every
    other coordinate full. Scales: none, 0 (the whole table is 0), r - 1 and a full element."""
    r = C.ints_to_mont([(0, 1, O.R_MOD - 1)[i % 3] for i in range(n)])
    if pattern == "stage_zero":
        r[n - 11:n - 8] = 0
        r[:n - 11] = rand_limbs_full(0xED + n, n - 11)
    for sc in (None, C.ints_to_mont([0])[0], C.ints_to_mont([O.R_MOD - 1])[0], rand_limbs_full(0xEE, 1)[0]):
        got = EqPolynomial.evals(sess, r, sc).evals()
        want = C.eq_evals(r, sc, threads=4 if n > 12 else 1)
        assert (got == want).all()
        if sc is not None and not sc.any():
            assert not got.any()


@pytest.mark.parametrize("kind", ["full254", "challenge125", "mixed", "wide_hi4", "wide_hi4_stage"])
def test_eq_2pow22(sess, kind):
    """BASELINE size; the point as full elements, as 125-bit challenges [0,0,lo,hi] (the 4-row product
    path, mod.rs:172-184), and mixed; then [0,0,x,y] with y across the top limb's whole canonical range, everywhere
    or only on the three register-stage variables r[11..14) that decide the streaming kernel's hi4 path."""
    n = 22
    r = rand_limbs(0xE0, n)
    if kind in ("challenge125", "mixed"):
        r[:, 0] = 0
        r[:, 1] = 0
        r[:, 3] &= np.uint64((1 << 61) - 1)
    if kind == "mixed":
        r[12] = rand_limbs(5, 1)[0]
    if kind == "wide_hi4":
        r = wide_hi4(0xE1, n)
    if kind == "wide_hi4_stage":
        r = rand_limbs_full(0xE2, n)
        r[11:14] = wide_hi4(0xE3, 3)
    got = EqPolynomial.evals(sess, r).evals()
    want = C.eq_evals(r, None, threads=C.max_threads())
    assert (got == want).all()
