"""Shared helpers for the -m gpu parity tests (CUDA path through the C ABI vs the oracle)."""
import numpy as np

from oracle import bn254 as O
from oracle import coracle as C



from oracle.coracle import rand_challenge, rand_limbs  # noqa: E402,F401


def rand_full(seed: int) -> np.ndarray:
    return np.array(O.to_mont_limbs(O.random_fr(seed, 1)[0]), dtype=np.uint64)


EDGE_INTS = [0, 1, 2, O.R_MOD - 1, O.R_MOD - 2, (1 << 256) % O.R_MOD, (1 << 64) - 1, (1 << 128) - 1, (1 << 253) + 5]


def edge_ints(p: int) -> list[int]:
    """EDGE_INTS reduced mod p plus the edges of p itself: p - 1, p - 2 and 2^256 mod p."""
    return [e % p for e in EDGE_INTS] + [p - 1, p - 2, (1 << 256) % p]


# ---- operand families that drive the kernels to the bounds their comments argue ------------------------------
# Every family returns raw Montgomery limbs (n, 4) of canonical elements: the value the limbs spell is < p.
# rand_limbs never sets the top 3 bits, so the top third of Fr never shows up in it.

def limbs_of(raw: int) -> np.ndarray:
    """The four u64 limbs of a raw 256-bit integer (no Montgomery conversion)."""
    return np.array([(raw >> (64 * k)) & ((1 << 64) - 1) for k in range(4)], dtype=np.uint64)


def limbs_below(a: np.ndarray, bound: int) -> np.ndarray:
    """Row mask: the raw integer of a[i] < bound (limb-wise, most significant first)."""
    b = limbs_of(bound)
    lt = np.zeros(a.shape[0], dtype=bool)
    eq = np.ones(a.shape[0], dtype=bool)
    for k in (3, 2, 1, 0):
        lt |= eq & (a[:, k] < b[k])
        eq &= a[:, k] == b[k]
    return lt


def rand_limbs_full(seed: int, n: int, p: int = O.R_MOD) -> np.ndarray:
    """Raw limbs uniform over [0, p), by rejection: the top limb is drawn from [0, p >> 192] and the rows whose
    value lands at or above p are drawn again."""
    rng = np.random.Generator(np.random.PCG64(seed))
    top = np.uint64(p >> 192)
    a = np.empty((n, 4), dtype=np.uint64)
    todo = np.arange(n)
    while todo.size:
        d = rng.integers(0, 1 << 64, size=(todo.size, 4), dtype=np.uint64)
        d[:, 3] = rng.integers(0, int(top) + 1, size=todo.size, dtype=np.uint64)
        a[todo] = d
        todo = todo[~limbs_below(d, p)]
    return a


def top_band(seed: int, n: int, p: int = O.R_MOD) -> np.ndarray:
    """Raw limbs uniform over [p - 2^128, p): r - 1 - u for a uniform 128-bit u, every operand near p."""
    rng = np.random.Generator(np.random.PCG64(seed))
    u = rng.integers(0, 1 << 64, size=(n, 2), dtype=np.uint64)
    pm1 = limbs_of(p - 1)
    a = np.empty((n, 4), dtype=np.uint64)
    a[:, 0] = pm1[0] - u[:, 0]
    b0 = (u[:, 0] > pm1[0]).astype(np.uint64)
    a[:, 1] = pm1[1] - u[:, 1] - b0
    b1 = ((u[:, 1] > pm1[1]) | ((u[:, 1] == pm1[1]) & (b0 == 1))).astype(np.uint64)
    a[:, 2] = pm1[2] - b1
    b2 = ((pm1[2] == 0) & (b1 == 1)).astype(np.uint64)
    a[:, 3] = pm1[3] - b2
    return a


R_MINUS_1 = limbs_of(O.R_MOD - 1)
CH_ZERO = np.zeros(4, dtype=np.uint64)                        # all-zero limbs: the 4-row product path
CH_ONE = np.array(O.to_mont_limbs(1), dtype=np.uint64)        # the Montgomery one: the full product


def parity_table(n: int, invert: bool = False) -> np.ndarray:
    """2^n entries, T[x] = raw r - 1 where popcount(x) is odd (even with invert), else 0. Bound with challenges
    0 and 1 only, it stays a (possibly inverted) parity table in every round and both orders, so every pair is
    (0, r - 1) or (r - 1, 0) and the lazy difference hi + p - lo is 2p - 1 or 1 in every round."""
    odd = (np.bitwise_count(np.arange(1 << n, dtype=np.uint64)) & 1).astype(bool)
    return const_table(n, O.R_MOD - 1) * (odd != invert)[:, None].astype(np.uint64)


def const_table(n: int, raw: int) -> np.ndarray:
    """2^n copies of the raw limbs of `raw`: 0 makes every sum and claim 0, r - 1 makes every difference 0."""
    return np.tile(limbs_of(raw), (1 << n, 1))


def wide_hi4(seed: int, n: int | None = None) -> np.ndarray:
    """A canonical multiplier [0, 0, x, y] (the 4-row product path) with x a full limb and y uniform below r's top
    limb - the whole legal range, not the 61-bit mask of a 125-bit challenge. n=None: one element (4,)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    k = 1 if n is None else n
    a = np.zeros((k, 4), dtype=np.uint64)
    a[:, 2] = rng.integers(0, 1 << 64, size=k, dtype=np.uint64)
    a[:, 3] = rng.integers(0, O.R_MOD >> 192, size=k, dtype=np.uint64)
    return a[0] if n is None else a
