"""Sumcheck members over products of 5..8 tables, and split-eq members over 4..8 tables (degree up to 9): every round
and the final evaluations against the threaded C oracle, limb for limb, in both binding orders, with the operand
families of gpu_util (whole field, the band just below r, parity tables, constant tables) and challenges that take
both bind paths (125-bit, full 254-bit, and [0, 0, x, y] across the top limb's whole range). Also verify mode, a first
round without a claim, the shapes that stay rejected, and batches: through the device RoundScheduler (degree <= 7)
and through the sequential fallback prove_batch takes for a member of degree 8 or 9."""
import numpy as np
import pytest

import jolt_b200
from jolt_b200 import (HIGH_TO_LOW, LOW_TO_HIGH, BatchMember, EqProductMember, Polynomial, ProductMember,
                       RoundScheduler, SumcheckError)
from jolt_b200 import _lib
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import (CH_ONE, CH_ZERO, const_table, parity_table, rand_challenge, rand_full, rand_limbs_full, top_band,
                      wide_hi4)

pytestmark = pytest.mark.gpu

ORDERS = [HIGH_TO_LOW, LOW_TO_HIGH]
FAMILIES = ["full", "top", "parity", "parity_alt", "zero", "rmax"]
C_SWEEP_MAX_TABLES = 8  # the C oracle's round sweep takes products of at most 8 tables


@pytest.fixture(scope="module")
def sess():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.fixture(scope="module")
def sess_verify():
    """a context that computes s(1) on the device and checks s(0) + s(1) against the claim (no SKIP1)"""
    s = jolt_b200.Session(0)
    s.set_verify_rounds(True)
    yield s
    s.close()


def round_evals(tabs, degree, order, thr):
    """s(0..degree) of sum_x prod_j tabs[j](x). Up to 8 tables this is the C oracle's sweep. With more (the split-eq
    oracle of m = 8 materialises eq as a ninth table) each s(t) is a full sum over the tables bound at the challenge
    t: the first two bound tables are folded into one by the oracle's field product, and the sweep's s(0) + s(1)
    over the remaining 8 is the sum of their product over every entry."""
    if len(tabs) <= C_SWEEP_MAX_TABLES:
        return C.mont_to_ints(C.product_round_evals(tabs, degree, order, thr))
    n = tabs[0].shape[0]
    out = []
    for t in range(degree + 1):
        tl = np.array(O.to_mont_limbs(t), dtype=np.uint64)
        b = [C.bind(x, tl, order, thr) for x in tabs]
        b = [C.f_vec(0, 2, b[0], b[1])] + b[2:]
        if n == 2:  # one entry left: no sweep
            out.append(int(np.prod([C.mont_to_ints(x)[0] for x in b], dtype=object)) % O.R_MOD)
        else:
            s01 = C.mont_to_ints(C.product_round_evals(b, 1, order, thr))
            out.append((s01[0] + s01[1]) % O.R_MOD)
    return out


class CMember:
    """The oracle side of one product member: sum_x prod_j T[j](x) over the threaded C oracle, with O.prove_batch's
    member interface (challenges as ints) and bind() for challenge limbs."""

    def __init__(self, tabs, order):
        self.cur, self.degree, self.order = list(tabs), len(tabs), order
        self.thr = C.max_threads()

    def evals(self):
        return round_evals(self.cur, self.degree, self.order, self.thr)

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


def prove_every_round(mem, ref, chs, with_claim=True):
    """Drives the device member and its oracle through every round with the same challenges: each round's evaluations
    and, after the last bind, the final evaluations limb for limb."""
    bind = None
    for rnd in range(mem.num_rounds()):
        if bind is not None:
            ref.bind(bind)
        want = ref.evals()
        claim = (want[0] + want[1]) % O.R_MOD if (with_claim or rnd > 0) else None
        got = mem.prove_round_evals(bind, rnd, claim)
        assert got == want, f"round {rnd}: first difference at t = {next(t for t, (a, b) in enumerate(zip(got, want)) if a != b)}"
        bind = chs[rnd]
    ref.bind(bind)
    mem.finish_rounds(bind)


def product_member(sess, tabs, order):
    return ProductMember(sess, [Polynomial.new(sess, t) for t in tabs], order)


# ---- ProductMember, m = 5..8 --------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("n", [14, 18])
@pytest.mark.parametrize("m", [5, 6, 7, 8])
def test_product_every_round(sess, m, n, order):
    tabs = make_tables("full", m, n, 0x8100 + 16 * m + n)
    mem = product_member(sess, tabs, order)
    assert mem.degree() == m and mem.num_rounds() == n
    ref = CMember(tabs, order)
    prove_every_round(mem, ref, make_challenges("full", n, 0x8200 + m))
    assert mem.final_evals() == ref.final_evals()
    mem.close()


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("m", [5, 8])
def test_product_families_every_round(sess, m, order, family):
    n = 16
    tabs = make_tables(family, m, n, 0x8300 + 16 * m)
    mem = product_member(sess, tabs, order)
    ref = CMember(tabs, order)
    prove_every_round(mem, ref, make_challenges(family, n, 0x8400 + m))
    assert mem.final_evals() == ref.final_evals()
    mem.close()


@pytest.mark.parametrize("order", ORDERS)
def test_product_m8_2pow20_every_round(sess, order):
    """2^19 pairs in round 0: every thread carries several pair indices"""
    n = 20
    tabs = make_tables("full", 8, n, 0x8500)
    mem = product_member(sess, tabs, order)
    ref = CMember(tabs, order)
    prove_every_round(mem, ref, make_challenges("full", n, 0x8600))
    assert mem.final_evals() == ref.final_evals()
    mem.close()


def test_product_m8_2pow22_parity_every_round(sess):
    """Eight parity tables: every root product is r - 1 times r - 1 or 0 on the same pairs in every round, so a thread's
    17-word accumulator gathers many products of ~2^508"""
    n = 22
    tabs = make_tables("parity", 8, n, 0)
    mem = product_member(sess, tabs, HIGH_TO_LOW)
    ref = CMember(tabs, HIGH_TO_LOW)
    prove_every_round(mem, ref, make_challenges("parity", n, 0x8722))
    assert mem.final_evals() == ref.final_evals()
    mem.close()


# ---- EqProductMember, m = 4..8: the oracle materialises eq(w, .) * scale as one more table ------------------------
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("n,scaled", [(18, False), (20, True)], ids=["2pow18", "2pow20-scaled"])
@pytest.mark.parametrize("m", [4, 5, 6, 7, 8])
def test_eq_member_every_round(sess, m, n, scaled, order):
    tabs = make_tables("full", m, n, 0x8800 + 16 * m + n)
    w = rand_limbs_full(0x8900 + n, n)
    scale = rand_full(0x8a00 + m) if scaled else None
    mem = EqProductMember(sess, [Polynomial.new(sess, t) for t in tabs], w, scale, order=order)
    assert mem.num_rounds() == n and mem.degree() == m + 1
    ref = CMember([C.eq_evals(w, scale, C.max_threads())] + tabs, order)
    prove_every_round(mem, ref, make_challenges("full", n, 0x8b00 + m))
    fe = ref.final_evals()
    assert mem.final_evals() == fe[1:]
    assert mem.eq_scalar() == fe[0]
    mem.close()


# ---- modes and misuse ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("m", [5, 8])
def test_verify_mode_every_round(sess_verify, m, order):
    """no SKIP1: the device computes s(1) as well, and the claim is checked"""
    n = 14
    tabs = make_tables("full", m, n, 0x8c00 + m)
    mem = product_member(sess_verify, tabs, order)
    ref = CMember(tabs, order)
    prove_every_round(mem, ref, make_challenges("full", n, 0x8d00 + m))
    assert mem.final_evals() == ref.final_evals()
    mem.close()


def test_verify_mode_wrong_claim_raises(sess_verify):
    n = 12
    tabs = make_tables("full", 7, n, 0x8e00)
    mem = product_member(sess_verify, tabs, HIGH_TO_LOW)
    want = CMember(tabs, HIGH_TO_LOW).evals()
    with pytest.raises(SumcheckError):
        mem.prove_round_evals(None, 0, (want[0] + want[1] + 1) % O.R_MOD)
    mem.close()


@pytest.mark.parametrize("order", ORDERS)
def test_first_round_without_claim(sess, order):
    n = 14
    tabs = make_tables("full", 6, n, 0x8f00)
    mem = product_member(sess, tabs, order)
    ref = CMember(tabs, order)
    prove_every_round(mem, ref, make_challenges("full", n, 0x9000), with_claim=False)
    assert mem.final_evals() == ref.final_evals()
    mem.close()


def test_nine_tables_rejected(sess):
    n = 6
    with pytest.raises(jolt_b200.JoltB200Error) as e:
        ProductMember(sess, [Polynomial.new(sess, t) for t in make_tables("full", 9, n, 0x9100)])
    assert e.value.status == _lib.JB_ERR_UNSUPPORTED
    with pytest.raises(jolt_b200.JoltB200Error) as e:
        EqProductMember(sess, [Polynomial.new(sess, t) for t in make_tables("full", 9, n, 0x9200)],
                        rand_limbs_full(0x9300, n))
    assert e.value.status == _lib.JB_ERR_UNSUPPORTED


# ---- batches ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
def test_batch_with_degree8_member(sess, order):
    """A degree-8 product, a split-eq m = 6 (degree 7) and an m = 2 product with ragged windows: the degree-8 member does
    not fit the scheduler's 8 evaluations per work item, so prove_batch runs the members in declaration order."""
    windows = [(14, 2), (16, 0), (15, 1)]
    max_vars = 16
    tabs8 = make_tables("full", 8, 14, 0x9400)
    tabs_eq = make_tables("full", 6, 16, 0x9500)
    w = rand_limbs_full(0x9600, 16)
    scale = rand_full(0x9601)
    tabs2 = make_tables("full", 2, 15, 0x9700)
    refs = [CMember(tabs8, order), CMember([C.eq_evals(w, scale, C.max_threads())] + tabs_eq, order),
            CMember(tabs2, order)]
    desc, total = [], 0
    for i, (ln, off) in enumerate(windows):
        ev = refs[i].evals()
        claim = (ev[0] + ev[1]) % O.R_MOD
        coeff = O.random_fr(0x9800 + i, 1)[0]
        desc.append(dict(input_claim=claim, coefficient=coeff, rounds=ln, offset=off))
        total = (total + coeff * claim * pow(2, max_vars - ln, O.R_MOD)) % O.R_MOD
    kinds = (rand_challenge, rand_full, wide_hi4)
    pts = [O.from_mont_limbs(kinds[r % 3](0x9900 + r)) for r in range(max_vars)]
    want = O.prove_batch(desc, refs, max_vars, 8, total, lambda r, c: pts[r])
    mems = [product_member(sess, tabs8, order),
            EqProductMember(sess, [Polynomial.new(sess, t) for t in tabs_eq], w, scale, order=order),
            product_member(sess, tabs2, order)]
    got = jolt_b200.prove_batch_native([BatchMember(**d) for d in desc], mems, max_vars, 8, total,
                                       lambda r, poly: pts[r])
    assert [p.coefficients for p in got.round_polynomials] == want["round_polys"]
    assert got.challenges == want["challenges"] and got.final_claim == want["final_claim"]
    assert got.member_claims == want["member_claims"]
    fe = [r.final_evals() for r in refs]
    assert mems[0].final_evals() == fe[0]
    assert mems[1].final_evals() == fe[1][1:] and mems[1].eq_scalar() == fe[1][0]
    assert mems[2].final_evals() == fe[2]
    for m in mems:
        m.close()


@pytest.mark.parametrize("order", ORDERS)
def test_scheduler_heterogeneous_degree7_batch(sess, order):
    """m = 5 and m = 7 products through the device RoundScheduler (overlapped launches): each member's round polynomial
    in every round and its final evaluations equal the member's own oracle"""
    n = 14
    tabs = [make_tables("full", 5, n, 0x9a00), make_tables("full", 7, n, 0x9b00)]
    refs = [CMember(t, order) for t in tabs]
    mems = [product_member(sess, t, order) for t in tabs]
    sched = RoundScheduler(sess, mems)
    chs = make_challenges("full", n, 0x9c00)
    bind = None
    for rnd in range(n):
        work, want = [], []
        for i, ref in enumerate(refs):
            if bind is not None:
                ref.bind(bind)
            ev = ref.evals()
            want.append(O.uni_from_evals(ev))
            work.append((i, rnd, bind, (ev[0] + ev[1]) % O.R_MOD))
        got = sched.batch_prove_round(work)
        assert [p.coefficients for p in got] == want, f"round {rnd}"
        bind = chs[rnd]
    for ref in refs:
        ref.bind(bind)
    sched.batch_finish_rounds([(0, bind), (1, bind)])
    for mem, ref in zip(mems, refs):
        assert mem.final_evals() == ref.final_evals()
    sched.close()
    for m in mems:
        m.close()


def test_scheduler_rejects_degree8_members(sess):
    n = 8
    prod8 = product_member(sess, make_tables("full", 8, n, 0x9d00), HIGH_TO_LOW)
    eq7 = EqProductMember(sess, [Polynomial.new(sess, t) for t in make_tables("full", 7, n, 0x9e00)],
                          rand_limbs_full(0x9f00, n))
    for mem in (prod8, eq7):
        with pytest.raises(jolt_b200.JoltB200Error) as e:
            RoundScheduler(sess, [mem])
        assert e.value.status == _lib.JB_ERR_UNSUPPORTED
        mem.close()
