"""Device Fr/Fq add/sub/mul vs the oracle, bit-exact (mirrors bn254_differential.rs:75-99 at scale)."""
import numpy as np
import pytest

import jolt_b200
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import EDGE_INTS, edge_ints, limbs_of, rand_limbs, rand_limbs_full, wide_hi4

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sess():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.mark.parametrize("fld,p", [(0, O.R_MOD), (1, O.Q_MOD)])
def test_vec_ops_bit_exact(sess, fld, p):
    n = 1 << 20
    # first half raw < 2^253 < both moduli (canonical for Fr and Fq), second half uniform over [0, p): the top third
    # of the field, which the first half never reaches
    a = np.concatenate([rand_limbs(11 + fld, n // 2), rand_limbs_full(33 + fld, n // 2, p)])
    b = np.concatenate([rand_limbs(22 + fld, n // 2), rand_limbs_full(44 + fld, n // 2, p)])
    # the edges in Montgomery form (incl. p - 1, p - 2 and 2^256 mod p of THIS field), then raw limbs p - 1 and p - 2
    edge = np.vstack([C.ints_to_mont(edge_ints(p), p), limbs_of(p - 1), limbs_of(p - 2)])
    k = len(edge)
    # all edge x edge pairs up front
    a[: k * k] = np.repeat(edge, k, axis=0)
    b[: k * k] = np.tile(edge, (k, 1))
    for op in (0, 1, 2):
        got = sess.vec_op(fld, op, a, b)
        want = C.f_vec(fld, op, a, b)
        assert (got == want).all(), f"field {fld} op {op}: {(got != want).any(axis=1).sum()} mismatches"
    # neg and square (bn254_differential.rs:75-99 also pins these): -a == 0 - a, a^2 == a * a
    assert (sess.vec_op(fld, 4, a, b) == C.f_vec(fld, 1, np.zeros_like(a), a)).all()
    assert (sess.vec_op(fld, 5, a, b) == C.f_vec(fld, 2, a, a)).all()


def test_mul_by_challenge_limbs(sess):
    # montmul(a, [0,0,lo,hi]) via the 4-row path == generic Montgomery product: the 125-bit challenge (hi masked to
    # 61 bits), then hi drawn across the top limb's whole canonical range against whole-field operands
    n = 1 << 16
    a = rand_limbs(5, n)
    b = rand_limbs(6, n)
    b[:, 0] = 0
    b[:, 1] = 0
    b[:, 3] &= np.uint64((1 << 61) - 1)
    a[:9] = C.ints_to_mont(EDGE_INTS)
    a_full = rand_limbs_full(7, n)
    a_full[:12] = C.ints_to_mont(edge_ints(O.R_MOD))
    for a, b in ((a, b), (a_full, wide_hi4(8, n))):
        got = sess.vec_op(0, 3, a, b)
        assert (got == C.f_vec(0, 2, a, b)).all()
        assert (sess.vec_op(0, 2, a, b) == got).all()
