"""G1 MSM on the device vs the oracle (mirrors crates/jolt-crypto/tests/group_laws.rs:12-146 and
SURVEY.md Appendix B): msm == naive sum (n <= 2^10), == oracle Pippenger (larger n), edge cases.
G1/MSM parity is unpinned by golden vectors (the reference holds none): results are compared as
affine (x, y) integers against the oracle."""
import numpy as np
import pytest

import jolt_b200
from jolt_b200 import G1Bases, Polynomial, g1_affine_limbs, g1_jacobian_to_affine
from oracle import bn254 as O
from oracle import coracle as C
from gpu_util import rand_limbs

pytestmark = pytest.mark.gpu

G = np.array(O.to_mont_limbs(1, O.Q_MOD) + O.to_mont_limbs(2, O.Q_MOD), dtype=np.uint64)


@pytest.fixture(scope="module")
def sess():
    s = jolt_b200.Session(0)
    yield s
    s.close()


@pytest.fixture(scope="module")
def srs_bases():
    """SRS-like bases beta^i * G (scheme.rs:54-73), 2^14 of them, from the C oracle."""
    beta = C.ints_to_mont([O.random_fr(0x4D534D, 1)[0]])[0]
    return C.g1_powers(1 << 14, G, beta)


def oracle_affine(xy, inf):
    return None if inf else (O.from_mont_limbs(xy[:4], O.Q_MOD), O.from_mont_limbs(xy[4:], O.Q_MOD))


@pytest.mark.parametrize("n", [1, 2, 3, 17, 64, 257, 1024])
def test_msm_matches_naive(sess, srs_bases, n):
    sc = rand_limbs(0x5CA1A2 + n, n)
    got = g1_jacobian_to_affine(G1Bases.from_affine(sess, srs_bases[:n]).msm(sc))
    assert got == oracle_affine(*C.g1_msm_naive(srs_bases[:n], sc))
    assert O.g1_is_on_curve(got)


@pytest.mark.parametrize("n", [1 << 12, 1 << 14])
def test_msm_matches_oracle_pippenger(sess, srs_bases, n):
    sc = rand_limbs(0x5CA1A2 + n, n)
    bases = G1Bases.from_affine(sess, srs_bases[:n])
    want = oracle_affine(*C.g1_msm_pippenger(srs_bases[:n], sc, 0, C.max_threads()))
    assert g1_jacobian_to_affine(bases.msm(sc)) == want
    # scalars already on the device (a folded HyperKZG polynomial): same value
    assert g1_jacobian_to_affine(bases.msm(Polynomial.new(sess, sc))) == want
    # offset windows of the SRS (kzg_commit uses g1_powers[..len])
    half = n // 2
    want2 = oracle_affine(*C.g1_msm_pippenger(srs_bases[half:n], sc[:half], 0, C.max_threads()))
    assert g1_jacobian_to_affine(bases.msm(sc[:half], offset=half)) == want2


def test_msm_empty_single_and_mismatch(sess, srs_bases):
    bases = G1Bases.from_affine(sess, srs_bases[:8])
    assert g1_jacobian_to_affine(bases.msm(np.zeros((0, 4), dtype=np.uint64))) is None          # group_laws.rs:143
    k = O.random_fr(3, 1)[0]
    one = g1_jacobian_to_affine(bases.msm(C.ints_to_mont([k])))                                  # group_laws.rs:135
    assert one == O.g1_scalar_mul(O.G1_GEN, k)
    with pytest.raises(jolt_b200.JoltB200Error, match="length mismatch"):                        # mod.rs:200-204
        bases.msm(rand_limbs(1, 9))
    with pytest.raises(jolt_b200.JoltB200Error, match="length mismatch"):
        jolt_b200.msm(sess, srs_bases[:4], rand_limbs(1, 5))


def test_msm_edge_scalars_and_bases(sess):
    # zero scalars, scalar 1 and r-1, repeated bases, P and -P with equal scalars, identity bases
    pts = [O.g1_scalar_mul(O.G1_GEN, k) for k in (1, 2, 3, 5, 7, 11, 13, 17)]
    pts[2] = pts[1]                      # repeated base -> the doubling branch inside a bucket
    pts[4] = O.g1_neg(pts[3])            # P and -P
    pts[6] = None                        # identity base
    sc = [0, 1, 1, 12345, 12345, O.R_MOD - 1, 999, (1 << 253) + 7]
    want = O.g1_msm_naive(pts, sc)
    got = g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs(pts), C.ints_to_mont(sc)))
    assert got == want
    # all-zero scalars and all-cancelling terms give the identity
    assert g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs(pts), C.ints_to_mont([0] * 8))) is None
    assert g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs([pts[3], pts[4]]), C.ints_to_mont([77, 77]))) is None
    # many copies of one base with one scalar: every term lands in the same buckets (P + P doubling chain)
    n = 300
    got = g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs([pts[0]] * n), C.ints_to_mont([5] * n)))
    assert got == O.g1_scalar_mul(O.G1_GEN, 5 * n)


def test_msm_small_scalars_u64(sess, srs_bases):
    # the msm_u64 shape of the legacy facade (jolt-prover-legacy/src/msm/mod.rs:35-79): small integers
    n = 1 << 10
    vals = [(i * 2654435761) % (1 << 32) for i in range(n)]
    sc = C.ints_to_mont(vals)
    want = oracle_affine(*C.g1_msm_pippenger(srs_bases[:n], sc, 0, C.max_threads()))
    assert g1_jacobian_to_affine(G1Bases.from_affine(sess, srs_bases[:n]).msm(sc)) == want


def test_jacobian_upload_normalises(sess):
    pts = [O.g1_scalar_mul(O.G1_GEN, k) for k in (3, 9, 27)]
    zs = O.random_fr(5, 3, O.Q_MOD)
    jac = np.zeros((4, 12), dtype=np.uint64)
    for i, ((x, y), z) in enumerate(zip(pts, zs)):
        jac[i, :4] = O.to_mont_limbs(x * z * z % O.Q_MOD, O.Q_MOD)
        jac[i, 4:8] = O.to_mont_limbs(y * z * z * z % O.Q_MOD, O.Q_MOD)
        jac[i, 8:] = O.to_mont_limbs(z, O.Q_MOD)
    jac[3, :4] = O.to_mont_limbs(1, O.Q_MOD)
    jac[3, 4:8] = O.to_mont_limbs(1, O.Q_MOD)          # (1, 1, 0): the identity
    bases = G1Bases.from_jacobian(sess, jac)
    assert (bases.affine() == g1_affine_limbs(pts + [None])).all()
    sc = [2, 3, 4, 5]
    assert g1_jacobian_to_affine(bases.msm(C.ints_to_mont(sc))) == O.g1_msm_naive(pts + [None], sc)


def test_msm_linearity_large(sess, srs_bases):
    """Size-independent property at 2^14 (homomorphism, commit_open_verify.rs:131-188):
    msm(a*s + b*t) == a*msm(s) + b*msm(t)."""
    n = 1 << 14
    s, t = rand_limbs(1, n), rand_limbs(2, n)
    a, b = O.random_fr(3, 2)
    A = np.tile(C.ints_to_mont([a]), (n, 1))
    Bm = np.tile(C.ints_to_mont([b]), (n, 1))
    comb = C.f_vec(0, 0, C.f_vec(0, 2, s, A), C.f_vec(0, 2, t, Bm))
    bases = G1Bases.from_affine(sess, srs_bases)
    lhs = g1_jacobian_to_affine(bases.msm(comb))
    ps, pt = g1_jacobian_to_affine(bases.msm(s)), g1_jacobian_to_affine(bases.msm(t))
    rhs = O.g1_add(O.g1_scalar_mul(ps, a), O.g1_scalar_mul(pt, b))
    assert lhs == rhs


def _weighted_sum(sc_limbs: np.ndarray) -> int:
    """sum_i s_i * (i + 1) mod r from Montgomery limbs, vectorised over 32-bit words."""
    a = np.ascontiguousarray(sc_limbs, dtype=np.uint64).reshape(-1, 4)
    n = a.shape[0]
    wts = np.arange(1, n + 1, dtype=object)
    total = 0
    for limb in range(4):
        for half in range(2):
            words = ((a[:, limb] >> np.uint64(32 * half)) & np.uint64(0xFFFFFFFF)).astype(object)
            total += int((words * wts).sum()) << (64 * limb + 32 * half)
    return total * pow(1 << 256, -1, O.R_MOD) % O.R_MOD


def test_generated_multiples_are_multiples(sess):
    bases = G1Bases.generate_multiples(sess, G, 100)
    xy = bases.affine()
    for i in (0, 1, 31, 32, 33, 63, 64, 99):
        assert oracle_affine(xy[i], False) == O.g1_scalar_mul(O.G1_GEN, i + 1)


@pytest.mark.parametrize("log_n", [16, 20])
def test_msm_closed_form_at_scale(sess, log_n):
    """BASELINE config 3 size (2^20): bases (i+1)*G make the MSM a single scalar multiplication,
    msm(s) == (sum_i s_i (i+1)) * G - an exact, size-independent check."""
    n = 1 << log_n
    bases = G1Bases.generate_multiples(sess, G, n)
    sc = rand_limbs(0x5CA1A2, n)
    got = g1_jacobian_to_affine(bases.msm(sc))
    assert got == O.g1_scalar_mul(O.G1_GEN, _weighted_sum(sc))


def test_msm_skewed_digits(sess):
    """Every scalar equal: each window has ONE non-empty bucket holding all n points - the worst case
    for a bucket-per-thread schedule; the chunked task plan must still be exact (and not crawl)."""
    n = 1 << 14
    bases = G1Bases.generate_multiples(sess, G, n)
    k = O.random_fr(77, 1)[0]
    sc = np.tile(C.ints_to_mont([k]), (n, 1))
    got = g1_jacobian_to_affine(bases.msm(sc))
    assert got == O.g1_scalar_mul(O.G1_GEN, k * (n * (n + 1) // 2) % O.R_MOD)
    # 0/1 scalars (a flag polynomial): only the digit-1 bucket of window 0 is populated
    bits = np.array([(i * 7 + 3) % 5 == 0 for i in range(n)])
    sc = C.ints_to_mont([int(b) for b in bits])
    got = g1_jacobian_to_affine(bases.msm(sc))
    assert got == O.g1_scalar_mul(O.G1_GEN, int(sum(i + 1 for i in range(n) if bits[i])))


@pytest.mark.parametrize("window_bits", [0, 10, 13])
def test_msm_precomputed_windows_same_value(sess, srs_bases, window_bits):
    """jb_srs_precompute: shared-bucket MSM over 2^(c w) P_i == per-window MSM == oracle."""
    n = 1 << 14
    sc = rand_limbs(0x5CA1A2 + 99, n)
    want = oracle_affine(*C.g1_msm_pippenger(srs_bases[:n], sc, 0, C.max_threads()))
    plain = G1Bases.from_affine(sess, srs_bases[:n])
    pre = G1Bases.from_affine(sess, srs_bases[:n]).precompute(window_bits)
    assert g1_jacobian_to_affine(plain.msm(sc)) == want
    assert g1_jacobian_to_affine(pre.msm(sc)) == want
    half = n // 2          # offset window of the SRS, still on the shared path
    want2 = oracle_affine(*C.g1_msm_pippenger(srs_bases[half:n], sc[:half], 0, C.max_threads()))
    assert g1_jacobian_to_affine(pre.msm(sc[:half], offset=half)) == want2
    small = rand_limbs(5, 16)   # a small MSM over the same handle takes the plain path
    assert g1_jacobian_to_affine(pre.msm(small)) == oracle_affine(*C.g1_msm_naive(srs_bases[:16], small))


def test_msm_precomputed_edge_cases(sess):
    pts = [O.g1_scalar_mul(O.G1_GEN, k) for k in (1, 2, 3, 5, 7, 11, 13, 17)] * 64
    pts[6] = None
    sc = ([0, 1, 1, 12345, 12345, O.R_MOD - 1, 999, (1 << 253) + 7] * 64)
    pts[4] = O.g1_neg(pts[3])
    bases = G1Bases.from_affine(sess, g1_affine_limbs(pts)).precompute(9)
    want = O.g1_msm_naive(pts, sc)
    assert g1_jacobian_to_affine(bases.msm(C.ints_to_mont(sc))) == want


def test_msm_precomputed_closed_form_2pow20(sess):
    n = 1 << 20
    bases = G1Bases.generate_multiples(sess, G, n).precompute()
    sc = rand_limbs(0x5CA1A2, n)
    assert g1_jacobian_to_affine(bases.msm(sc)) == O.g1_scalar_mul(O.G1_GEN, _weighted_sum(sc))


@pytest.mark.parametrize("n", [1, 2, 5, 33, 1000, 4096])
def test_small_msm_over_precomputed_srs(sess, srs_bases, n):
    """n <= 4096 over a precomputed handle takes the 8-bit-window table (no doubling chains)."""
    bases = G1Bases.from_affine(sess, srs_bases[: 1 << 13]).precompute()
    sc = rand_limbs(31 + n, n)
    want = oracle_affine(*C.g1_msm_pippenger(srs_bases[:n], sc, 0, C.max_threads()))
    assert g1_jacobian_to_affine(bases.msm(sc)) == want
    off = 100
    want2 = oracle_affine(*C.g1_msm_pippenger(srs_bases[off:off + n], sc, 0, C.max_threads()))
    assert g1_jacobian_to_affine(bases.msm(sc, offset=off)) == want2


def test_msm_exceptional_inputs(sess):
    """What the reference's batch addition excludes by precondition and an MSM cannot: equal points in a bucket (tangent),
    opposite points (identity result), identity bases, all terms in one bucket."""
    n = 1 << 13
    # every base the same point, every scalar the same: each bucket is a list of n copies of one point
    one = [O.g1_scalar_mul(O.G1_GEN, 9)] * n
    got = g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs(one), C.ints_to_mont([5] * n)))
    assert got == O.g1_scalar_mul(O.G1_GEN, 9 * 5 * n)
    # P, -P alternating with one scalar: every pair cancels
    P = O.g1_scalar_mul(O.G1_GEN, 31)
    alt = [P if i % 2 == 0 else O.g1_neg(P) for i in range(n)]
    assert g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs(alt), C.ints_to_mont([77] * n))) is None
    # a few distinct multiples repeated, identity bases mixed in, a handful of distinct scalars (crowded buckets,
    # sums of pairs that coincide with other sums: (1 + 4) G == (2 + 3) G)
    ks = [1, 2, 3, 4, 5, 6, 7, 8]
    pts = [O.g1_scalar_mul(O.G1_GEN, k) for k in ks]
    bases, mult = [], []
    for i in range(n):
        if i % 11 == 0:
            bases.append(None)
            mult.append(0)
        else:
            bases.append(pts[i % 8])
            mult.append(ks[i % 8])
    svals = [O.random_fr(5, 4)[i % 4] for i in range(n)]
    total = sum(m * s for m, s in zip(mult, svals)) % O.R_MOD
    got = g1_jacobian_to_affine(jolt_b200.msm(sess, g1_affine_limbs(bases), C.ints_to_mont(svals)))
    assert got == O.g1_scalar_mul(O.G1_GEN, total)
    # closed form over (i + 1) G with uniform scalars at 2^16, plain and precomputed
    n = 1 << 16
    gen = G1Bases.generate_multiples(sess, G, n)
    sc = rand_limbs(0x5CA1A2, n)
    want = O.g1_scalar_mul(O.G1_GEN, _weighted_sum(sc))
    assert g1_jacobian_to_affine(gen.msm(sc)) == want
    gen.precompute()
    assert g1_jacobian_to_affine(gen.msm(sc)) == want
    gen.free()
