"""Every round of every sumcheck member shape against the threaded C oracle, at sizes where a thread carries several
pairs, with operands at the edges the kernels' bounds allow: the whole field, a band just below r, parity tables whose
lazy differences are 2p - 1 in every round, constant tables, and challenges that take both product paths (125-bit,
full 254-bit, and [0, 0, x, y] with y across the top limb's whole range). Each member runs under the default session
(resident kernel, lookahead, thin passes) and under one that launches a kernel per round."""
import os

import numpy as np
import pytest

import jolt_b200
from jolt_b200 import (HIGH_TO_LOW, LOW_TO_HIGH, BatchMember, EqProductMember, Polynomial, ProductMember,
                       SumOfProductsMember)
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import (CH_ONE, CH_ZERO, const_table, parity_table, rand_challenge, rand_full, rand_limbs_full, top_band,
                      wide_hi4)

pytestmark = pytest.mark.gpu

ORDERS = [HIGH_TO_LOW, LOW_TO_HIGH]


@pytest.fixture(scope="module")
def sess_resident():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.fixture(scope="module")
def sess_launch():
    """a context with the resident service off: one kernel launch per round all the way down"""
    os.environ["JB_NO_TAIL"] = "1"
    try:
        s = jolt_b200.Session(0)
    finally:
        del os.environ["JB_NO_TAIL"]
    s.per_round = True
    yield s
    s.close()


@pytest.fixture(params=["resident", "launch"])
def sess(request):
    return request.getfixturevalue("sess_" + request.param)


def check_launches(sess, launches, n):
    """the default session proves a whole product or sum-of-products sumcheck with ONE resident kernel launch"""
    if getattr(sess, "per_round", False):
        assert launches >= n, launches
    else:
        assert launches == 1, launches


class CMember:
    """The oracle side of one member: sum_x sum_k prod_j T[k * degree + j](x) over the threaded C oracle, with
    O.prove_batch's member interface (challenges as ints) and bind() for challenge limbs."""

    def __init__(self, tabs, degree, order):
        self.cur, self.degree, self.order = list(tabs), degree, order
        self.thr = C.max_threads()

    def evals(self):
        d = self.degree
        terms = [C.mont_to_ints(C.product_round_evals(self.cur[k:k + d], d, self.order, self.thr))
                 for k in range(0, len(self.cur), d)]
        return [sum(v) % O.R_MOD for v in zip(*terms)]

    def bind(self, r_limbs):
        self.cur = [C.bind(t, r_limbs, self.order, self.thr) for t in self.cur]

    def prove_round(self, bind_c, rnd, claim):
        if bind_c is not None:
            self.finish_rounds(bind_c)
        ev = self.evals()
        assert (ev[0] + ev[1]) % O.R_MOD == claim % O.R_MOD, f"oracle round {rnd}: the batch claim is not honest"
        return O.uni_from_evals(ev)

    def finish_rounds(self, bind_c):
        self.bind(np.array(O.to_mont_limbs(bind_c % O.R_MOD), dtype=np.uint64))

    def final_evals(self):
        return [C.mont_to_ints(t)[0] for t in self.cur]


FAMILIES = ["full", "top", "parity", "parity_alt", "zero", "rmax"]


def make_tables(family, count, n, seed):
    if family == "full":
        return [rand_limbs_full(seed + j, 1 << n) for j in range(count)]
    if family == "top":
        return [top_band(seed + j, 1 << n) for j in range(count)]
    if family == "parity":
        return [parity_table(n) for _ in range(count)]
    if family == "parity_alt":
        return [parity_table(n, invert=j % 2 == 1) for j in range(count)]
    return [const_table(n, 0 if family == "zero" else O.R_MOD - 1) for _ in range(count)]


def make_challenges(family, n, seed):
    """parity tables: challenges 0 and 1 only (both in every run); otherwise 125-bit, full 254-bit and wide [0,0,x,y]
    in turn"""
    if family.startswith("parity"):
        bits = np.random.Generator(np.random.PCG64(seed)).integers(0, 2, size=n)
        bits[:2] = (0, 1)
        return [CH_ONE if b else CH_ZERO for b in bits]
    kinds = (rand_challenge, rand_full, wide_hi4)
    return [kinds[i % 3](seed + i) for i in range(n)]


def prove_every_round(sess, mem, ref, chs):
    """Drives the device member and its oracle through every round with the same challenges: each round's evaluations
    and the final evaluations limb for limb. Returns the launches the device made."""
    n = mem.num_rounds()
    l0 = sess.launch_count
    bind = None
    for rnd in range(n):
        if bind is not None:
            ref.bind(bind)
        want = ref.evals()
        got = mem.prove_round_evals(bind, rnd, (want[0] + want[1]) % O.R_MOD)
        assert got == want, f"round {rnd}: first difference at t = {next(t for t, (a, b) in enumerate(zip(got, want)) if a != b)}"
        bind = chs[rnd]
    ref.bind(bind)
    mem.finish_rounds(bind)
    return sess.launch_count - l0



# ---- ProductMember ----------------------------------------------------------------------------------------------
# 2^18 is thin from round 0 under the resident kernel; 2^20 runs generic rounds first, then thin ones.
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("m,n", [(1, 18), (2, 18), (3, 18), (4, 18), (2, 20)])
def test_product_member_every_round(sess, m, n, order, family):
    tabs = make_tables(family, m, n, 0x5100 + 16 * m + n)
    mem = ProductMember(sess, [Polynomial.new(sess, t) for t in tabs], order)
    ref = CMember(tabs, m, order)
    launches = prove_every_round(sess, mem, ref, make_challenges(family, n, 0x6100 + m))
    assert mem.final_evals() == ref.final_evals()
    mem.close()
    check_launches(sess, launches, n)


@pytest.mark.parametrize("order", ORDERS)
def test_product_member_2pow22_parity_every_round(sess_resident, order):
    """Two plain parity tables: both lazy differences are 2p - 1 on the same pairs in every round, so each pair adds
    an s(inf) product of up to (2p - 1)^2 ~ 2^509 and a thread's 17-word accumulator, carrying many pairs, passes
    2^512 - its carry into the top word decides the round."""
    n = 22
    tabs = make_tables("parity", 2, n, 0)
    mem = ProductMember(sess_resident, [Polynomial.new(sess_resident, t) for t in tabs], order)
    ref = CMember(tabs, 2, order)
    launches = prove_every_round(sess_resident, mem, ref, make_challenges("parity", n, 0x6222))
    assert mem.final_evals() == ref.final_evals()
    mem.close()
    check_launches(sess_resident, launches, n)


# ---- SumOfProductsMember 2 x 2 ----------------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["full", "parity"])
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("n", [18, 20])
def test_sum_of_products_every_round(sess, n, order, family):
    tabs = make_tables(family, 4, n, 0x5300 + n)
    mem = SumOfProductsMember(sess, [Polynomial.new(sess, t) for t in tabs], 2, 2, order)
    ref = CMember(tabs, 2, order)
    launches = prove_every_round(sess, mem, ref, make_challenges(family, n, 0x6300 + n))
    assert mem.final_evals() == ref.final_evals()
    mem.close()
    check_launches(sess, launches, n)


# ---- EqProductMember: the oracle materialises eq(w, .) * scale as one more table ---------------------------------
@pytest.mark.parametrize("family", ["full", "parity"])
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("n", [18, 20])
@pytest.mark.parametrize("m", [1, 2, 3])
def test_eq_member_every_round(sess, m, n, order, family):
    tabs = make_tables(family, m, n, 0x5400 + 16 * m + n)
    w = rand_limbs_full(0x77 + n, n)
    scale = rand_full(0x78 + m) if family == "full" else None
    mem = EqProductMember(sess, [Polynomial.new(sess, t) for t in tabs], w, scale, order=order)
    assert mem.num_rounds() == n and mem.degree() == m + 1
    ref = CMember([C.eq_evals(w, scale, C.max_threads())] + tabs, m + 1, order)
    prove_every_round(sess, mem, ref, make_challenges(family, n, 0x6400 + m))
    fe = ref.final_evals()
    assert mem.final_evals() == fe[1:]
    assert mem.eq_scalar() == fe[0]
    mem.close()


# ---- RoundScheduler through prove_batch_native: homogeneous batches with ragged lengths and offsets ---------------
@pytest.mark.parametrize("shape", [
    (3, 1, [(16, 0), (14, 2), (15, 1)]),     # three m = 3 products: one resident kernel with D = 3
    (4, 1, [(15, 1), (16, 0), (14, 2)]),     # three m = 4 products: D = 4
    (2, 2, [(16, 0), (15, 1), (14, 2)]),     # three 2 x 2 sums of products
], ids=["m3", "m4", "sop2x2"])
@pytest.mark.parametrize("order", ORDERS)
def test_scheduler_homogeneous_batch_every_round(sess_resident, shape, order):
    """(rounds, offset) windows all end at the last round: a member joins the batch once the rounds before its window
    have halved its scaled claim back to its own"""
    sess = sess_resident
    degree, terms, windows = shape
    max_vars = max(ln + off for ln, off in windows)
    tabs = [make_tables("full", degree * terms, ln, 0x5500 + 64 * i + 8 * degree + terms) for i, (ln, _) in enumerate(windows)]
    refs = [CMember(t, degree, order) for t in tabs]
    desc, total = [], 0
    for i, (ln, off) in enumerate(windows):
        ev = refs[i].evals()
        claim = (ev[0] + ev[1]) % O.R_MOD
        coeff = O.random_fr(0x5600 + i, 1)[0]
        desc.append(dict(input_claim=claim, coefficient=coeff, rounds=ln, offset=off))
        total = (total + coeff * claim * pow(2, max_vars - ln, O.R_MOD)) % O.R_MOD
    kinds = (rand_challenge, rand_full, wide_hi4)
    pts = [O.from_mont_limbs(kinds[r % 3](0x5700 + r)) for r in range(max_vars)]
    want = O.prove_batch(desc, refs, max_vars, degree, total, lambda r, c: pts[r])
    if terms == 1:
        mems = [ProductMember(sess, [Polynomial.new(sess, t) for t in tb], order) for tb in tabs]
    else:
        mems = [SumOfProductsMember(sess, [Polynomial.new(sess, t) for t in tb], degree, terms, order) for tb in tabs]
    l0 = sess.launch_count
    got = jolt_b200.prove_batch_native([BatchMember(**d) for d in desc], mems, max_vars, degree, total,
                                       lambda r, poly: pts[r])
    launches = sess.launch_count - l0
    assert [p.coefficients for p in got.round_polynomials] == want["round_polys"]
    assert got.challenges == want["challenges"] and got.final_claim == want["final_claim"]
    assert got.member_claims == want["member_claims"]
    for mem, ref in zip(mems, refs):
        assert mem.final_evals() == ref.final_evals()
        mem.close()
    assert launches == 1, launches     # the whole batch was ONE kernel launch
