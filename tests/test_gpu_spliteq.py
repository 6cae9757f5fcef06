"""Split-eq (Gruen) member on the device: sum_x eq(w, x) prod_j f_j(x) without materialising eq
(crates/jolt-poly/src/split_eq.rs). Oracle: the plain (m+1)-table product sumcheck over the materialised eq
table - the round polynomials are the same field values (Gruen's factorisation is a schedule, not a relation)."""
import numpy as np
import pytest

import jolt_b200
from jolt_b200 import BatchMember, EqPolynomial, EqProductMember, HIGH_TO_LOW, LOW_TO_HIGH, Polynomial, ProductMember
from jolt_b200 import field as F
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import rand_challenge

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sess():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.mark.parametrize("order", [LOW_TO_HIGH, HIGH_TO_LOW])
@pytest.mark.parametrize("m", [1, 2, 3])
@pytest.mark.parametrize("n", [1, 2, 3, 5, 9, 12])
def test_eq_member_lockstep_vs_oracle(sess, m, n, order):
    tabs = [O.random_fr(300 + 10 * m + j, 1 << n) for j in range(m)]
    w = O.random_fr(77 + n, n)
    eq_tab = O.eq_evals(w)                                    # r[0] <-> MSB (eq.rs:218-219)
    ref = O.ProductMember([eq_tab] + tabs, order)
    gpu = EqProductMember(sess, [Polynomial.from_ints(sess, t) for t in tabs], C.ints_to_mont(w), order=order)
    assert gpu.num_rounds() == n and gpu.degree() == m + 1
    claim = sum(eq_tab[i] * int(np.prod([t[i] for t in tabs], dtype=object)) for i in range(1 << n)) % O.R_MOD
    ch = O.random_fr(5, n)
    bind = None
    for rnd in range(n):
        want = ref.prove_round(bind, rnd, claim)
        got = gpu.prove_round(bind, rnd, claim)
        assert got.coefficients == want, f"round {rnd}"
        bind = ch[rnd]
        claim = got.evaluate(bind)
    ref.finish_rounds(bind)
    gpu.finish_rounds(bind)
    fe = ref.final_evals()
    assert gpu.final_evals() == fe[1:]
    assert gpu.eq_scalar() == fe[0]                          # eq(w, r) with the order's challenge-to-variable map
    assert gpu.eq_scalar() * int(np.prod(gpu.final_evals(), dtype=object)) % O.R_MOD == claim


def test_eq_member_scaled_and_challenge_point(sess):
    n, m = 8, 2
    tabs = [O.random_fr(900 + j, 1 << n) for j in range(m)]
    w_limbs = np.stack([rand_challenge(40 + i) for i in range(n)])       # 125-bit challenge point
    w = F.limbs_to_ints(w_limbs)
    scale = O.random_fr(3, 1)[0]
    eq_tab = O.eq_evals(w, scale)
    ref = O.ProductMember([eq_tab] + tabs, O.LOW_TO_HIGH)
    gpu = EqProductMember(sess, [Polynomial.from_ints(sess, t) for t in tabs], w_limbs, scale)
    claim = sum(e * a * b for e, a, b in zip(eq_tab, *tabs)) % O.R_MOD
    bind = None
    for rnd in range(n):
        want = ref.prove_round(bind, rnd, claim)
        got = gpu.prove_round(bind, rnd, claim)
        assert got.coefficients == want
        bind = F.from_limbs(rand_challenge(60 + rnd))
        claim = got.evaluate(bind)


def test_eq_member_in_the_engine_and_errors(sess):
    n, m = 10, 2
    tabs = [O.random_fr(11 + j, 1 << n) for j in range(m)]
    w = O.random_fr(9, n)
    eq_tab = O.eq_evals(w)
    claim = sum(e * a * b for e, a, b in zip(eq_tab, *tabs)) % O.R_MOD
    mem = EqProductMember(sess, [Polynomial.from_ints(sess, t) for t in tabs], C.ints_to_mont(w))
    res = jolt_b200.prove_batch_native([BatchMember(claim, 1, n, 0)], [mem], n, m + 1, claim, seed=5)
    # same proof from the plain member over the materialised eq table
    plain = ProductMember(sess, [EqPolynomial.evals(sess, C.ints_to_mont(w))] + [Polynomial.from_ints(sess, t) for t in tabs],
                          LOW_TO_HIGH)
    res2 = jolt_b200.prove_batch_native([BatchMember(claim, 1, n, 0)], [plain], n, m + 1, claim, seed=5)
    assert res.challenges == res2.challenges and res.final_claim == res2.final_claim
    assert [p.coefficients for p in res.round_polynomials] == [p.coefficients for p in res2.round_polynomials]
    assert mem.eq_scalar() == plain.final_evals()[0]
    fresh = EqProductMember(sess, [Polynomial.from_ints(sess, tabs[0])], C.ints_to_mont(w))
    with pytest.raises(jolt_b200.JoltB200Error, match="claim is required"):
        fresh.prove_round_evals(None, 0, None)
    with pytest.raises(jolt_b200.JoltB200Error, match="point length"):
        EqProductMember(sess, [Polynomial.from_ints(sess, tabs[0])], C.ints_to_mont(w[:-1]))


@pytest.mark.parametrize("order", [LOW_TO_HIGH, HIGH_TO_LOW])
@pytest.mark.parametrize("case", ["w_zero_first", "scale_zero", "w_zero_round2"])
def test_eq_member_noninvertible_round_is_an_error(sess, order, case):
    """The Gruen round divides by l1 = scale * eq-so-far * w_c: a round whose l1 is zero (w_c = 0, or scale = 0) is an
    error, not a wrong round polynomial. The rounds before it still match the oracle."""
    n, m = 6, 2
    tabs = [O.random_fr(40 + j, 1 << n) for j in range(m)]
    w = O.random_fr(41, n)
    bad_round = 2 if case == "w_zero_round2" else 0
    if case != "scale_zero":
        w[bad_round if order == HIGH_TO_LOW else n - 1 - bad_round] = 0   # the variable round k binds
    scale = 0 if case == "scale_zero" else None
    eq_tab = O.eq_evals(w, scale)
    ref = O.ProductMember([eq_tab] + tabs, order)
    gpu = EqProductMember(sess, [Polynomial.from_ints(sess, t) for t in tabs], C.ints_to_mont(w), scale, order=order)
    claim = sum(e * a * b for e, a, b in zip(eq_tab, *tabs)) % O.R_MOD
    ch = O.random_fr(42, n)
    bind = None
    for rnd in range(bad_round):
        want = ref.prove_round(bind, rnd, claim)
        got = gpu.prove_round(bind, rnd, claim)
        assert got.coefficients == want, f"round {rnd}"
        bind = ch[rnd]
        claim = got.evaluate(bind)
    with pytest.raises(jolt_b200.JoltB200Error, match="must be invertible"):
        gpu.prove_round_evals(bind, bad_round, claim)
