"""Python mirror of the reference's operator surface for the hot path, over the C ABI.

Names, argument meaning and error behaviour follow the reference so that the parity tests read
like its own (crates/jolt-poly/src/dense.rs, eq.rs, univariate.rs; crates/jolt-sumcheck/src/prover.rs).
All table-sized data stays on the device; only O(rounds * degree) values cross back."""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field as dc_field

import numpy as np

from . import _lib
from . import field as F
from ._lib import JoltB200Error, c_u64p

HIGH_TO_LOW = 0  # BindingOrder::HighToLow - pairs (i, i + half)
LOW_TO_HIGH = 1  # BindingOrder::LowToHigh - pairs (2i, 2i + 1)


def _p(a: np.ndarray):
    assert a.dtype == np.uint64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_u64p)


def _limbs(x) -> np.ndarray:
    """Accepts a Python int (canonical value) or 4 Montgomery limbs."""
    if isinstance(x, (int, np.integer)):
        return F.to_limbs(int(x))
    a = np.ascontiguousarray(x, dtype=np.uint64).reshape(-1)
    assert a.size == 4, "field element = 4 x u64 Montgomery limbs"
    return a


class SumcheckError(RuntimeError):
    """Mirrors jolt_sumcheck::SumcheckError (crates/jolt-sumcheck/src/error.rs)."""


class Session:
    """Device half of ProofSession (crates/jolt-kernels/src/backend.rs:283-286)."""

    def __init__(self, device: int = 0, cuda_stream: int | None = None):
        self.lib = _lib.load()
        h = ctypes.c_void_p()
        if cuda_stream is None:
            st = self.lib.jb_ctx_create(device, ctypes.byref(h))
        else:
            st = self.lib.jb_ctx_create_on_stream(device, ctypes.c_void_p(cuda_stream), ctypes.byref(h))
        if st != _lib.JB_OK:
            raise JoltB200Error(st, self.lib.jb_status_str(st).decode())
        self.h = h
        self.device = device

    def check(self, st: int):
        if st != _lib.JB_OK:
            detail = self.lib.jb_last_error(self.h).decode() or self.lib.jb_status_str(st).decode()
            if st == _lib.JB_ERR_ROUND_CHECK:
                raise SumcheckError(detail)
            raise JoltB200Error(st, detail)

    def synchronize(self):
        self.check(self.lib.jb_ctx_synchronize(self.h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.jb_ctx_launch_count(self.h))

    def set_verify_rounds(self, on: bool = True):
        """on: members compute s(1) and check s(0)+s(1)==claim (reference tier, naive.rs:301-308);
        off (default): s(1) = claim - s(0) (optimized tier, support.rs:450-460)."""
        self.check(self.lib.jb_ctx_set_verify_rounds(self.h, 1 if on else 0))

    def timing_enable(self, on: bool = True, min_items: int = 0):
        self.check(self.lib.jb_ctx_timing_enable(self.h, 1 if on else 0, min_items))

    def timing_collect(self, cap: int = 4096) -> list[dict]:
        kinds = (ctypes.c_int * cap)()
        items = (ctypes.c_uint64 * cap)()
        ms_m = (ctypes.c_int * cap)()
        ms = (ctypes.c_double * cap)()
        cnt = ctypes.c_size_t()
        self.check(self.lib.jb_ctx_timing_collect(self.h, kinds, items, ms_m, ms, cap, ctypes.byref(cnt)))
        names = {0: "fused_bind_eval", 1: "bind", 2: "eval_only", 3: "eq", 4: "msm_accumulate"}
        return [dict(kind=names.get(kinds[i], str(kinds[i])), items=int(items[i]), m=int(ms_m[i]), ms=float(ms[i]))
                for i in range(cnt.value)]

    def close(self):
        if self.h:
            self.lib.jb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # element-wise parity harness (bn254_differential.rs:75-99)
    def vec_op(self, field: int, op: int, a: np.ndarray, b: np.ndarray) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
        b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 4)
        out = np.empty_like(a)
        self.check(self.lib.jb_vec_op(self.h, field, op, _p(a), _p(b), _p(out), a.shape[0]))
        return out


# jb_scalar_kind (include/jolt_b200.h): compact-table / small-scalar encodings
SCALAR_KINDS = {"fr": 0, "u8": 1, "u16": 2, "u32": 3, "u64": 4, "u128": 5, "i64": 6, "i128": 7, "s64": 8, "s128": 9}
_DTYPE_KIND = {np.dtype(np.uint8): "u8", np.dtype(np.bool_): "u8", np.dtype(np.uint16): "u16",
               np.dtype(np.uint32): "u32", np.dtype(np.uint64): "u64", np.dtype(np.int64): "i64"}


def small_scalars(values, kind: str | None = None) -> tuple[np.ndarray, int, int]:
    """(contiguous byte-exact array, jb_scalar_kind, n) for a primitive integer column. `values`: a numpy
    array of dtype bool/u8/u16/u32/u64/i64, or - for the 128-bit kinds - a sequence of Python ints with
    `kind` = "u128" / "i128" (stored as 16 little-endian bytes each, two's complement). The sign-magnitude kinds
    "s64" / "s128" (jolt_field::signed::S64 / S128, crates/jolt-field/src/signed.rs:25-32) take a sequence of
    (magnitude, is_positive) tuples or of Python ints (sign taken from the int; (0, False) is the reference's -0)
    and are stored as jb_s64 / jb_s128 records: N u64 magnitude limbs, then the sign byte, padded to 8."""
    if kind in ("s64", "s128"):
        limbs = 1 if kind == "s64" else 2
        rec = np.zeros((len(values), limbs + 1), dtype=np.uint64)
        for i, v in enumerate(values):
            mag, pos = (abs(int(v)), int(v) >= 0) if not isinstance(v, (tuple, list)) else (int(v[0]), bool(v[1]))
            if not 0 <= mag < 1 << (64 * limbs):
                raise ValueError(f"{kind} magnitude out of range")
            for j in range(limbs):
                rec[i, j] = (mag >> (64 * j)) & 0xFFFFFFFFFFFFFFFF
            rec[i, limbs] = 1 if pos else 0  # little-endian: the sign byte is the first byte of the last word
        return rec, SCALAR_KINDS[kind], len(values)
    if kind in ("u128", "i128"):
        ints = [int(v) for v in values]
        lo_hi = np.empty((len(ints), 2), dtype=np.uint64)
        for i, v in enumerate(ints):
            if kind == "u128" and not 0 <= v < 1 << 128:
                raise ValueError("u128 value out of range")
            if kind == "i128" and not -(1 << 127) <= v < 1 << 127:
                raise ValueError("i128 value out of range")
            w = v & ((1 << 128) - 1)
            lo_hi[i, 0] = w & 0xFFFFFFFFFFFFFFFF
            lo_hi[i, 1] = w >> 64
        return lo_hi, SCALAR_KINDS[kind], len(ints)
    a = np.ascontiguousarray(values)
    name = _DTYPE_KIND.get(a.dtype)
    if name is None or (kind is not None and kind != name):
        raise ValueError(f"unsupported compact dtype {a.dtype} (kind={kind})")
    if a.dtype == np.bool_:
        a = a.astype(np.uint8)
    return a.reshape(-1), SCALAR_KINDS[name], a.size


class Polynomial:
    """Device-resident multilinear polynomial in evaluation form
    (jolt_poly::Polynomial<Fr>, dense.rs:35; legacy DensePolynomial, dense_mlpoly.rs:20)."""

    def __init__(self, session: Session, handle: int):
        self.s = session
        self.handle = handle

    @classmethod
    def new(cls, session: Session, evals_limbs: np.ndarray) -> "Polynomial":
        a = np.ascontiguousarray(evals_limbs, dtype=np.uint64).reshape(-1, 4)
        n = a.shape[0]
        if n == 0 or n & (n - 1):
            raise ValueError(f"Dense multi-linear polynomials must be made from a power of 2 (not {n})")
        h = ctypes.c_uint64()
        session.check(session.lib.jb_table_upload(session.h, _p(a), n, ctypes.byref(h)))
        return cls(session, h.value)

    @classmethod
    def from_ints(cls, session: Session, values) -> "Polynomial":
        return cls.new(session, F.ints_to_limbs(values))

    @classmethod
    def from_small(cls, session: Session, values, kind: str | None = None) -> "Polynomial":
        """Polynomial<T> for a primitive T (dense.rs:22-119) promoted to the field on the device
        (jb_table_upload_small): F::from(T), i.e. v mod r with negatives as r - |v|."""
        a, k, n = small_scalars(values, kind)
        if n == 0 or n & (n - 1):
            raise ValueError(f"Dense multi-linear polynomials must be made from a power of 2 (not {n})")
        h = ctypes.c_uint64()
        session.check(session.lib.jb_table_upload_small(session.h, a.ctypes.data_as(ctypes.c_void_p), n, k, ctypes.byref(h)))
        return cls(session, h.value)

    @classmethod
    def bind_to_field(cls, session: Session, values, scalar, order: int = HIGH_TO_LOW, kind: str | None = None) -> "Polynomial":
        """Polynomial<T>::bind_to_field (dense.rs:129-142): the compact table folded under `scalar` into a
        new field polynomial of half the length (fused promote + bind, jb_table_bind_small)."""
        a, k, n = small_scalars(values, kind)
        r = _limbs(scalar)
        h = ctypes.c_uint64()
        session.check(session.lib.jb_table_bind_small(session.h, a.ctypes.data_as(ctypes.c_void_p), n, k, _p(r), order,
                                                      ctypes.byref(h)))
        return cls(session, h.value)

    @classmethod
    def wrap_device(cls, session: Session, device_ptr: int, length: int) -> "Polynomial":
        h = ctypes.c_uint64()
        session.check(session.lib.jb_table_wrap_device(session.h, ctypes.c_void_p(device_ptr), length, ctypes.byref(h)))
        return cls(session, h.value)

    def __len__(self) -> int:
        n = ctypes.c_size_t()
        self.s.check(self.s.lib.jb_table_len(self.s.h, self.handle, ctypes.byref(n)))
        return n.value

    def num_vars(self) -> int:
        return len(self).bit_length() - 1

    def device_ptr(self) -> int:
        p = ctypes.c_void_p()
        self.s.check(self.s.lib.jb_table_device_ptr(self.s.h, self.handle, ctypes.byref(p)))
        return p.value

    def bind_with_order(self, scalar, order: int = HIGH_TO_LOW) -> None:
        r = _limbs(scalar)
        self.s.check(self.s.lib.jb_table_bind(self.s.h, self.handle, _p(r), order))

    def bind(self, scalar, order: int = HIGH_TO_LOW) -> None:
        """Polynomial::bind == HighToLow (dense.rs:169-171); the legacy signature passes the order."""
        self.bind_with_order(scalar, order)

    bind_parallel = bind  # legacy DensePolynomial::bind_parallel (dense_mlpoly.rs:78)

    def clone(self) -> "Polynomial":
        h = ctypes.c_uint64()
        self.s.check(self.s.lib.jb_table_clone(self.s.h, self.handle, ctypes.byref(h)))
        return Polynomial(self.s, h.value)

    def evals(self) -> np.ndarray:
        n = len(self)
        out = np.empty((n, 4), dtype=np.uint64)
        self.s.check(self.s.lib.jb_table_download(self.s.h, self.handle, _p(out), n))
        return out

    def to_ints(self) -> list[int]:
        return F.limbs_to_ints(self.evals())

    def free(self):
        if self.handle:
            self.s.check(self.s.lib.jb_table_free(self.s.h, self.handle))
            self.handle = 0


class EqPolynomial:
    """jolt_poly::EqPolynomial (eq.rs:24): tables in big-endian index order (r[0] <-> MSB)."""

    @staticmethod
    def evals(session: Session, r_limbs, scaling_factor=None) -> Polynomial:
        r = np.ascontiguousarray(r_limbs, dtype=np.uint64).reshape(-1, 4)
        sc = None if scaling_factor is None else _limbs(scaling_factor)
        h = ctypes.c_uint64()
        session.check(session.lib.jb_eq_evals(session.h, _p(r) if r.shape[0] else None, r.shape[0],
                                               _p(sc) if sc is not None else None, ctypes.byref(h)))
        return Polynomial(session, h.value)

    @staticmethod
    def evals_for_aligned_block(session: Session, r_limbs, start_index: int, block_size: int) -> Polynomial:
        r = np.ascontiguousarray(r_limbs, dtype=np.uint64).reshape(-1, 4)
        h = ctypes.c_uint64()
        session.check(session.lib.jb_eq_evals_aligned_block(session.h, _p(r), r.shape[0], start_index, block_size,
                                                             ctypes.byref(h)))
        return Polynomial(session, h.value)


class UnivariatePoly:
    """jolt_poly::UnivariatePoly (univariate.rs:27): coefficients ascending, values as ints mod r.
    Stays on the host in the reference too (O(d^2) work on <= ~10 elements)."""

    def __init__(self, coefficients: list[int]):
        self.coefficients = [c % F.R_MOD for c in coefficients]

    def degree(self) -> int:
        return max(len(self.coefficients) - 1, 0)

    def evaluate(self, point: int) -> int:
        acc = 0
        for c in reversed(self.coefficients):
            acc = (acc * point + c) % F.R_MOD
        return acc

    @classmethod
    def from_evals(cls, evals: list[int]) -> "UnivariatePoly":
        """Interpolation on nodes 0..n-1 (univariate.rs:198-202). Newton forward differences
        (exact in the field; value-equal to the reference's Vandermonde solve)."""
        p = F.R_MOD
        n = len(evals)
        diffs = [e % p for e in evals]
        newton = []
        for k in range(n):
            newton.append(diffs[0])
            diffs = [(diffs[i + 1] - diffs[i]) % p for i in range(len(diffs) - 1)]
        # p(x) = sum_k newton[k] * C(x, k); expand the falling factorials
        coeffs = [0] * n
        basis = [1]  # x(x-1)...(x-k+1) coefficients
        fact_inv = 1
        for k in range(n):
            if k:
                fact_inv = fact_inv * pow(k, -1, p) % p
            scale = newton[k] * fact_inv % p
            for i, b in enumerate(basis):
                coeffs[i] = (coeffs[i] + scale * b) % p
            nxt = [0] * (len(basis) + 1)
            for i, b in enumerate(basis):  # multiply by (x - k)
                nxt[i + 1] = (nxt[i + 1] + b) % p
                nxt[i] = (nxt[i] - k * b) % p
            basis = nxt
        return cls(coeffs)

    @classmethod
    def from_evals_and_hint(cls, hint: int, evals: list[int]) -> "UnivariatePoly":
        full = list(evals)
        full.insert(1, (hint - full[0]) % F.R_MOD)
        return cls.from_evals(full)

    def compress(self) -> list[int]:
        assert len(self.coefficients) >= 2, "cannot compress a polynomial of degree < 1"
        return self.coefficients[:1] + self.coefficients[2:]

    def __eq__(self, other):
        return isinstance(other, UnivariatePoly) and self.coefficients == other.coefficients

    def __repr__(self):
        return f"UnivariatePoly({[hex(c) for c in self.coefficients]})"


class ProductMember:
    """A device-backed ProveRounds member (prover.rs:52-72) for the relation
    sum_x prod_j f_j(x) over m = 1..8 dense tables, degree m - the GPU twin of the reference tier's
    NaiveSumcheckProver (naive.rs:241-316) / tests' DenseMember (tests.rs:1123-1175, m = 1). A RoundScheduler takes
    members of degree <= 7."""

    def __init__(self, session: Session, polys: list[Polynomial], order: int = HIGH_TO_LOW):
        self.s = session
        handles = np.array([p.handle for p in polys], dtype=np.uint64)
        h = ctypes.c_void_p()
        session.check(session.lib.jb_member_create(session.h, _p(handles), len(polys), order, ctypes.byref(h)))
        for p in polys:
            p.handle = 0  # ownership moved into the member
        self.h = h
        self.m = len(polys)

    def num_rounds(self) -> int:
        n = ctypes.c_size_t()
        self.s.check(self.s.lib.jb_member_num_rounds(self.h, ctypes.byref(n)))
        return n.value

    def degree(self) -> int:
        return self.m

    def prove_round_evals(self, bind, rnd: int, previous_claim=None) -> list[int]:
        b = None if bind is None else _limbs(bind)
        c = None if previous_claim is None else _limbs(previous_claim)
        out = np.empty((self.m + 1, 4), dtype=np.uint64)
        self.s.check(self.s.lib.jb_member_prove_round(self.h, _p(b) if b is not None else None, rnd,
                                                      _p(c) if c is not None else None, _p(out)))
        return F.limbs_to_ints(out)

    def prove_round(self, bind, rnd: int, previous_claim) -> UnivariatePoly:
        return UnivariatePoly.from_evals(self.prove_round_evals(bind, rnd, previous_claim))

    def finish_rounds(self, bind) -> None:
        self.s.check(self.s.lib.jb_member_finish_rounds(self.h, _p(_limbs(bind))))

    def final_evals(self, raw: bool = False):
        out = np.empty((self.m, 4), dtype=np.uint64)
        self.s.check(self.s.lib.jb_member_final_evals(self.h, _p(out)))
        return out if raw else F.limbs_to_ints(out)

    def close(self):
        if self.h:
            if self.s.h:  # (a member outliving its session was freed with the session's pools)
                self.s.lib.jb_member_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SumOfProductsMember(ProductMember):
    """ProveRounds member for sum_x sum_{k<terms} prod_{j<factors} f_{k*factors+j}(x) (jb_member_create_sop) - the
    shape of the reference's optimized claim-reduction kernels after paired-eq fusion, e.g. IncClaimReduction's
    A * RamInc + B * RdInc (crates/jolt-kernels/src/optimized/inc_claim_reduction.rs:47-203). `polys` in term-major
    order; degree = factors; final_evals() returns all factors * terms bound values."""

    def __init__(self, session: Session, polys: list[Polynomial], factors: int, terms: int, order: int = HIGH_TO_LOW):
        assert len(polys) == factors * terms
        self.s = session
        handles = np.array([p.handle for p in polys], dtype=np.uint64)
        h = ctypes.c_void_p()
        session.check(session.lib.jb_member_create_sop(session.h, _p(handles), factors, terms, order, ctypes.byref(h)))
        for p in polys:
            p.handle = 0
        self.h = h
        self.m = factors
        self.terms = terms

    def final_evals(self, raw: bool = False):
        out = np.empty((self.m * self.terms, 4), dtype=np.uint64)
        self.s.check(self.s.lib.jb_member_final_evals(self.h, _p(out)))
        return out if raw else F.limbs_to_ints(out)


class RoundScheduler:
    """Device traversal of a batch (jolt_sumcheck::RoundScheduler, prover.rs:106-120; jb_scheduler_*): every active
    member's round in one host round trip. `members`: ProductMember-likes of one session."""

    def __init__(self, session: Session, members: list):
        self.s = session
        self.members = list(members)
        arr = (ctypes.c_void_p * len(members))(*[m.h for m in members])
        h = ctypes.c_void_p()
        session.check(session.lib.jb_scheduler_create(session.h, arr, len(members), ctypes.byref(h)))
        self.h = h

    def batch_prove_round(self, work: list[tuple]) -> list[UnivariatePoly]:
        """work: [(member_index, local_round, bind_or_None, claim_or_None)] -> one round polynomial per item."""
        n = len(work)
        arr = (_lib.RoundWorkC * max(n, 1))()
        for i, (idx, rnd, bind, claim) in enumerate(work):
            arr[i].member, arr[i].round = idx, rnd
            arr[i].has_bind = 0 if bind is None else 1
            arr[i].has_claim = 0 if claim is None else 1
            if bind is not None:
                arr[i].bind[:] = [int(x) for x in _limbs(bind)]
            if claim is not None:
                arr[i].claim[:] = [int(x) for x in _limbs(claim)]
        out = np.zeros((max(n, 1), 8, 4), dtype=np.uint64)
        self.s.check(self.s.lib.jb_scheduler_prove_round(self.h, ctypes.cast(arr, ctypes.c_void_p), n, _p(out)))
        res = []
        for i, (idx, *_rest) in enumerate(work):
            d = self.members[idx].degree()
            res.append(UnivariatePoly.from_evals(F.limbs_to_ints(out[i, : d + 1])))
        return res

    def batch_finish_rounds(self, finishes: list[tuple]) -> None:
        """finishes: [(member_index, bind)]."""
        n = len(finishes)
        arr = (_lib.FinishWorkC * max(n, 1))()
        for i, (idx, bind) in enumerate(finishes):
            arr[i].member = idx
            arr[i].bind[:] = [int(x) for x in _limbs(bind)]
        self.s.check(self.s.lib.jb_scheduler_finish_rounds(self.h, ctypes.cast(arr, ctypes.c_void_p), n))

    def close(self):
        if self.h:
            self.s.lib.jb_scheduler_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EqProductMember(ProductMember):
    """ProveRounds member for sum_x eq(w, x) * prod_j f_j(x) (degree m + 1) with the eq polynomial kept
    split (GruenSplitEqPolynomial, crates/jolt-poly/src/split_eq.rs:159-447): no eq table is materialised,
    bound or streamed. `w_limbs`: n elements, w[0] <-> MSB; both binding orders (split_eq.rs:208-257). m = 1..8 tables
    (degree up to 9); a RoundScheduler takes members of degree <= 7, i.e. m <= 6."""

    def __init__(self, session: Session, polys: list[Polynomial], w_limbs, scale=None, order: int = LOW_TO_HIGH):
        self.s = session
        handles = np.array([p.handle for p in polys], dtype=np.uint64)
        w = np.ascontiguousarray(w_limbs, dtype=np.uint64).reshape(-1, 4)
        sc = None if scale is None else _limbs(scale)
        h = ctypes.c_void_p()
        session.check(session.lib.jb_eq_member_create(session.h, _p(handles), len(polys), _p(w), w.shape[0],
                                                      _p(sc) if sc is not None else None, order, ctypes.byref(h)))
        for p in polys:
            p.handle = 0
        self.h = h
        self.m = len(polys)

    def degree(self) -> int:
        return self.m + 1

    def prove_round_evals(self, bind, rnd: int, previous_claim=None) -> list[int]:
        b = None if bind is None else _limbs(bind)
        c = None if previous_claim is None else _limbs(previous_claim)
        out = np.empty((self.m + 2, 4), dtype=np.uint64)
        self.s.check(self.s.lib.jb_member_prove_round(self.h, _p(b) if b is not None else None, rnd,
                                                      _p(c) if c is not None else None, _p(out)))
        return F.limbs_to_ints(out)

    def eq_scalar(self) -> int:
        out = np.empty(4, dtype=np.uint64)
        self.s.check(self.s.lib.jb_eq_member_scalar(self.h, _p(out)))
        return F.from_limbs(out)


@dataclass
class BatchMember:
    """jolt_sumcheck::BatchMember (batch.rs:24-71)."""
    input_claim: int
    coefficient: int
    rounds: int
    offset: int = 0


@dataclass
class ProvedBatch:
    """prover.rs:153-157 (+ the per-round batched polynomials the recorder saw)."""
    challenges: list[int]
    final_claim: int
    member_claims: list[int]
    round_polynomials: list[UnivariatePoly] = dc_field(default_factory=list)


def prove_batch(members_desc: list[BatchMember], members: list, max_num_vars: int, max_degree: int, claimed_sum: int,
                absorb_round) -> ProvedBatch:
    """Host engine, line-for-line semantics of prove_batch (prover.rs:193-362); `absorb_round(round,
    UnivariatePoly) -> challenge` stands in for recorder.absorb_round + the transcript, which stay
    host-side (Fiat-Shamir is the only forced device sync per round, specs/clean-slate-prover.md:579-582)."""
    p = F.R_MOD
    if len(members) != len(members_desc):
        raise SumcheckError(f"BatchMemberCountMismatch {{ expected: {len(members_desc)}, got: {len(members)} }}")
    for i, (m, d) in enumerate(zip(members, members_desc)):
        if m.num_rounds() != d.rounds:
            raise SumcheckError(f"BatchMemberRoundsMismatch {{ member: {i}, expected: {d.rounds}, got: {m.num_rounds()} }}")
        if d.offset + d.rounds > max_num_vars:
            raise SumcheckError(f"BatchMemberWindowOutOfRange {{ member: {i} }}")
    if max_num_vars > 0 and max_degree < 1:
        raise SumcheckError(f"ZeroBatchDegree {{ max_num_vars: {max_num_vars} }}")
    two_inv = pow(2, -1, p)
    claims = [d.input_claim * pow(2, max_num_vars - d.rounds, p) % p for d in members_desc]
    running = claimed_sum % p
    challenges: list[int] = []
    pending: list[int | None] = [None] * len(members)
    polys: list[UnivariatePoly] = []
    for rnd in range(max_num_vars):
        batched = [0] * (max_degree + 1)
        work = []
        for i, (m, d) in enumerate(zip(members, members_desc)):
            active = d.offset <= rnd < d.offset + d.rounds
            if not active:
                claims[i] = claims[i] * two_inv % p
                batched[0] = (batched[0] + d.coefficient * claims[i]) % p
                continue
            b, pending[i] = pending[i], None
            work.append((i, m.prove_round(b, rnd - d.offset, claims[i])))
        for i, poly in work:
            if poly.degree() > max_degree:
                raise SumcheckError(f"DegreeBoundExceeded {{ got: {poly.degree()}, max: {max_degree} }}")
            for k, c in enumerate(poly.coefficients):
                batched[k] = (batched[k] + members_desc[i].coefficient * c) % p
        while len(batched) > 2 and batched[-1] == 0:  # trim_round_polynomial
            batched.pop()
        bp = UnivariatePoly(batched)
        if (bp.evaluate(0) + bp.evaluate(1)) % p != running:
            raise SumcheckError(f"RoundCheckFailed {{ round: {rnd} }}")
        c = absorb_round(rnd, bp) % p
        running = bp.evaluate(c)
        challenges.append(c)
        polys.append(bp)
        for i, poly in work:
            claims[i] = poly.evaluate(c)
            pending[i] = c
    for m, b in zip(members, pending):
        if b is not None:
            m.finish_rounds(b)
    return ProvedBatch(challenges, running, claims, polys)


def prove_batch_native(members_desc: list[BatchMember], members: list[ProductMember], max_num_vars: int,
                       max_degree: int, claimed_sum: int, absorb_round=None, seed: int = 0,
                       check_member_rounds: bool = True, raw: bool = False):
    """The same engine run by the C++ host layer (jolt_b200/csrc/sumcheck_host.cu) in one ABI call:
    no Python in the round loop. absorb_round=None uses the built-in SplitMix stand-in transcript
    (jb_absorb_round_splitmix125, seeded with `seed`)."""
    lib = _lib.load()
    n = len(members)
    desc = (_lib.BatchMemberC * n)()
    for i, d in enumerate(members_desc):
        desc[i].input_claim[:] = [int(x) for x in F.to_limbs(d.input_claim)]
        desc[i].coefficient[:] = [int(x) for x in F.to_limbs(d.coefficient)]
        desc[i].rounds = d.rounds
        desc[i].offset = d.offset
    handles = (ctypes.c_void_p * n)(*[m.h for m in members])
    seed_c = ctypes.c_uint64(seed)
    if absorb_round is None:
        fn = ctypes.cast(lib.jb_absorb_round_splitmix125, ctypes.c_void_p)
        user = ctypes.cast(ctypes.byref(seed_c), ctypes.c_void_p)
        keep = None
    else:
        def _cb(_user, rnd, coeffs, ncoeffs, out):
            poly = UnivariatePoly([F.from_limbs([coeffs[4 * k + i] for i in range(4)]) for k in range(ncoeffs)])
            c = F.to_limbs(absorb_round(rnd, poly))
            for i in range(4):
                out[i] = int(c[i])
            return 0
        keep = _lib.ABSORB_FN(_cb)
        fn = ctypes.cast(keep, ctypes.c_void_p)
        user = None
    ch = np.zeros((max_num_vars, 4), dtype=np.uint64)
    fin = np.zeros(4, dtype=np.uint64)
    mc = np.zeros((n, 4), dtype=np.uint64)
    rp = np.zeros((max_num_vars, max_degree + 1, 4), dtype=np.uint64)
    lens = (ctypes.c_size_t * max(max_num_vars, 1))()
    cs = F.to_limbs(claimed_sum)
    st = lib.jb_prove_batch(handles, ctypes.cast(desc, ctypes.c_void_p), n, max_num_vars, max_degree, _p(cs),
                            1 if check_member_rounds else 0, fn, user, _p(ch), _p(fin), _p(mc), _p(rp), lens)
    if st != _lib.JB_OK:
        sess = members[0].s
        detail = sess.lib.jb_last_error(sess.h).decode() or sess.lib.jb_status_str(st).decode()
        if st == _lib.JB_ERR_ROUND_CHECK:
            raise SumcheckError("RoundCheckFailed: " + detail)
        raise JoltB200Error(st, detail)
    if raw:  # the limb arrays as the ABI returned them (no big-int conversion on the caller's critical path)
        return ch, fin, mc, rp
    polys = [UnivariatePoly(F.limbs_to_ints(rp[r, : lens[r]])) for r in range(max_num_vars)]
    return ProvedBatch(F.limbs_to_ints(ch), F.from_limbs(fin), F.limbs_to_ints(mc), polys)


# ---- G1 / MSM ---------------------------------------------------------------------------------------
def g1_jacobian_to_affine(xyz_limbs) -> tuple[int, int] | None:
    """Host normalisation of the ABI's Jacobian result (x = X/Z^2, y = Y/Z^3); None = identity."""
    a = np.ascontiguousarray(xyz_limbs, dtype=np.uint64).reshape(3, 4)
    X, Y, Z = (F.from_limbs(a[i], F.Q_MOD) for i in range(3))
    if Z == 0:
        return None
    zi = pow(Z, -1, F.Q_MOD)
    return X * zi * zi % F.Q_MOD, Y * zi * zi * zi % F.Q_MOD


def g1_affine_limbs(points) -> np.ndarray:
    """[(x, y) | None] -> (n, 8) Montgomery limbs; the identity is x = y = 0."""
    out = np.zeros((len(points), 8), dtype=np.uint64)
    for i, P in enumerate(points):
        if P is not None:
            out[i, :4] = F.to_limbs(P[0], F.Q_MOD)
            out[i, 4:] = F.to_limbs(P[1], F.Q_MOD)
    return out


class G1Bases:
    """Device-resident affine G1 bases: the `bases: &[Bn254G1]` argument of JoltGroup::msm
    (crates/jolt-crypto/src/ec/group.rs:70) / HyperKZGProverSetup::g1_powers (scheme.rs:60-66),
    normalised once instead of per call (mod.rs:205)."""

    def __init__(self, session: Session, handle: int, n: int):
        self.s, self.handle, self.n = session, handle, n

    @classmethod
    def from_affine(cls, session: Session, xy_limbs: np.ndarray) -> "G1Bases":
        a = np.ascontiguousarray(xy_limbs, dtype=np.uint64).reshape(-1, 8)
        h = ctypes.c_uint64()
        session.check(session.lib.jb_srs_upload_affine(session.h, _p(a) if a.shape[0] else None, a.shape[0], ctypes.byref(h)))
        return cls(session, h.value, a.shape[0])

    @classmethod
    def from_jacobian(cls, session: Session, xyz_limbs: np.ndarray) -> "G1Bases":
        a = np.ascontiguousarray(xyz_limbs, dtype=np.uint64).reshape(-1, 12)
        h = ctypes.c_uint64()
        session.check(session.lib.jb_srs_upload_jacobian(session.h, _p(a) if a.shape[0] else None, a.shape[0], ctypes.byref(h)))
        return cls(session, h.value, a.shape[0])

    @classmethod
    def generate_multiples(cls, session: Session, base_xy_limbs: np.ndarray, n: int) -> "G1Bases":
        """bases[i] = (i + 1) * base, generated on the device (synthetic SRS for benches/tests)."""
        b = np.ascontiguousarray(base_xy_limbs, dtype=np.uint64).reshape(8)
        h = ctypes.c_uint64()
        session.check(session.lib.jb_srs_generate_multiples(session.h, _p(b), n, ctypes.byref(h)))
        return cls(session, h.value, n)

    def precompute(self, window_bits: int = 0) -> "G1Bases":
        """Builds the 2^(c w) * P_i table for a fixed SRS (jb_srs_precompute): later large MSMs over this
        handle share one bucket set across windows. Same group values."""
        self.s.check(self.s.lib.jb_srs_precompute(self.s.h, self.handle, window_bits))
        return self

    def __len__(self):
        n = ctypes.c_size_t()
        self.s.check(self.s.lib.jb_srs_len(self.s.h, self.handle, ctypes.byref(n)))
        return n.value

    def affine(self) -> np.ndarray:
        out = np.empty((self.n, 8), dtype=np.uint64)
        self.s.check(self.s.lib.jb_srs_download_affine(self.s.h, self.handle, _p(out), self.n))
        return out

    def msm(self, scalars, offset: int = 0) -> np.ndarray:
        """sum_i scalars[i] * bases[offset + i] as 12 Jacobian limbs. `scalars`: (n, 4) Montgomery
        limbs on the host, or a device-resident Polynomial. Length mismatch raises (mod.rs:200-204)."""
        out = np.zeros(12, dtype=np.uint64)
        if isinstance(scalars, Polynomial):
            n = len(scalars)
            self.s.check(self.s.lib.jb_msm_g1_table(self.s.h, self.handle, offset, scalars.handle, n, _p(out)))
        else:
            a = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
            self.s.check(self.s.lib.jb_msm_g1(self.s.h, self.handle, offset, _p(a) if a.shape[0] else None, a.shape[0], _p(out)))
        return out

    def msm_small(self, values, offset: int = 0, kind: str | None = None) -> np.ndarray:
        """VariableBaseMSM::msm_u8 .. msm_i128 (crates/jolt-prover-legacy/src/msm/mod.rs:90-150): the
        scalars are a primitive integer column (see small_scalars); 12 Jacobian limbs."""
        a, k, n = small_scalars(values, kind)
        out = np.zeros(12, dtype=np.uint64)
        self.s.check(self.s.lib.jb_msm_g1_small(self.s.h, self.handle, offset,
                                                a.ctypes.data_as(ctypes.c_void_p) if n else None, n, k, _p(out)))
        return out

    def batch_msm(self, columns) -> np.ndarray:
        """VariableBaseMSM::batch_msm / batch_msm_univariate (crates/jolt-prover-legacy/src/msm/mod.rs:160-181): one MSM
        per column against the PREFIX bases[..len(column)] of this base set. A column is (n, 4) Montgomery limbs
        (LargeScalars / UniPoly coefficients), a numpy integer array, or a (values, kind) pair as in small_scalars.
        Returns (len(columns), 12) Jacobian limbs."""
        keep, ptrs, lens, kinds = [], [], [], []
        for col in columns:
            if isinstance(col, tuple):
                a, k, n = small_scalars(col[0], col[1])
            elif isinstance(col, np.ndarray) and col.dtype == np.uint64 and col.ndim == 2 and col.shape[1] == 4:
                a, k, n = np.ascontiguousarray(col), SCALAR_KINDS["fr"], col.shape[0]
            else:
                a, k, n = small_scalars(col)
            keep.append(a)
            ptrs.append(a.ctypes.data if n else 0)
            lens.append(n)
            kinds.append(k)
        m = len(columns)
        out = np.zeros((max(m, 1), 12), dtype=np.uint64)
        self.s.check(self.s.lib.jb_msm_g1_batch(self.s.h, self.handle, m, (ctypes.c_void_p * max(m, 1))(*ptrs),
                                                (ctypes.c_size_t * max(m, 1))(*lens), (ctypes.c_int * max(m, 1))(*kinds), _p(out)))
        return out[:m]

    def msm_rows(self, values, rows: int, kind: str | None = None) -> np.ndarray:
        """Row-batched MSM (jb_msm_g1_rows): `values` is a row-major matrix of `rows` rows (a flat column as in
        small_scalars, or (rows * w, 4) Montgomery limbs with kind="fr"); every row is an MSM against bases[..w] -
        Dory's tier-1 row commitments (crates/jolt-dory/src/streaming.rs:53-201). Returns (rows, 12) Jacobian limbs."""
        if kind == "fr":
            a = np.ascontiguousarray(values, dtype=np.uint64).reshape(-1, 4)
            k, n = SCALAR_KINDS["fr"], a.shape[0]
        else:
            a, k, n = small_scalars(values, kind)
        if rows <= 0 or n % rows:
            raise ValueError("msm_rows: the number of scalars must be a multiple of rows")
        out = np.zeros((rows, 12), dtype=np.uint64)
        self.s.check(self.s.lib.jb_msm_g1_rows(self.s.h, self.handle, a.ctypes.data_as(ctypes.c_void_p) if n else None,
                                               rows, n // rows, k, _p(out)))
        return out

    def batch_add(self, index_sets) -> np.ndarray:
        """batch_g1_additions_multi_affine (crates/jolt-crypto/src/ec/bn254/batch_addition.rs:53-150): one affine
        sum (8 limbs; zeros = identity) per index set. Precondition: no pair of equal / opposite points."""
        offs = np.zeros(len(index_sets) + 1, dtype=np.uint64)
        for i, st in enumerate(index_sets):
            offs[i + 1] = offs[i] + len(st)
        flat = np.ascontiguousarray(np.concatenate([np.asarray(st, dtype=np.uint32) for st in index_sets]) if len(index_sets) and offs[-1]
                                    else np.zeros(0, dtype=np.uint32))
        out = np.zeros((max(len(index_sets), 1), 8), dtype=np.uint64)
        self.s.check(self.s.lib.jb_g1_batch_add(self.s.h, self.handle, _p(offs), flat.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)),
                                                len(index_sets), _p(out)))
        return out[: len(index_sets)]

    def msm_sharded(self, scalars, offset: int = 0) -> np.ndarray:
        """This rank's share of a term-partitioned MSM; every rank gets the same total (jb_msm_g1_sharded)."""
        out = np.zeros(12, dtype=np.uint64)
        a = np.ascontiguousarray(scalars, dtype=np.uint64).reshape(-1, 4)
        self.s.check(self.s.lib.jb_msm_g1_sharded(self.s.h, self.handle, offset, _p(a) if a.shape[0] else None, a.shape[0], _p(out)))
        return out

    def free(self):
        if self.handle:
            self.s.check(self.s.lib.jb_srs_free(self.s.h, self.handle))
            self.handle = 0


def msm(session: Session, bases_xy_limbs: np.ndarray, scalars_limbs: np.ndarray) -> np.ndarray:
    """JoltGroup::msm(bases, scalars): one-shot form (uploads the bases for this call)."""
    b = np.ascontiguousarray(bases_xy_limbs, dtype=np.uint64).reshape(-1, 8)
    s = np.ascontiguousarray(scalars_limbs, dtype=np.uint64).reshape(-1, 4)
    if b.shape[0] != s.shape[0]:
        raise JoltB200Error(_lib.JB_ERR_LENGTH, "msm: bases/scalars length mismatch")
    g = G1Bases.from_affine(session, b)
    try:
        return g.msm(s)
    finally:
        g.free()


# ---- HyperKZG prover side ------------------------------------------------------------------------
@dataclass
class HyperKZGProof:
    """jolt_hyperkzg::HyperKZGProof (types.rs): com = ell-1 intermediate commitments, w = 3 witness
    commitments (12 Jacobian limbs each), v[t][j] = f_j(u_t) as ints."""
    com: np.ndarray
    w: np.ndarray
    v: list[list[int]]


class HyperKZG:
    """HyperKZGScheme prover side (crates/jolt-hyperkzg/src/scheme.rs:275-338) over device-resident
    SRS powers (`G1Bases`) and polynomials."""

    @staticmethod
    def commit(bases: G1Bases, poly: Polynomial) -> np.ndarray:
        """CommitmentScheme::commit -> kzg_commit (kzg.rs:15-27): one MSM over g1_powers[..len]."""
        return bases.msm(poly)

    @staticmethod
    def open(bases: G1Bases, poly: Polynomial, point_limbs, challenge_r, challenge_q) -> HyperKZGProof:
        """HyperKZGScheme::open (scheme.rs:122-158). challenge_r(com (ell-1, 12) limbs) -> r and
        challenge_q(v [3][ell] ints) -> q stand in for the transcript (ints mod r)."""
        s = bases.s
        lib = s.lib
        pt = np.ascontiguousarray(point_limbs, dtype=np.uint64).reshape(-1, 4)
        ell = pt.shape[0]
        com = np.zeros((max(ell - 1, 1), 12), dtype=np.uint64)
        w = np.zeros((3, 12), dtype=np.uint64)
        v = np.zeros((3, max(ell, 1), 4), dtype=np.uint64)

        def _r(_user, com_ptr, ncom, out):
            arr = np.array([com_ptr[i] for i in range(ncom * 12)], dtype=np.uint64).reshape(ncom, 12)
            limbs = F.to_limbs(challenge_r(arr))
            for i in range(4):
                out[i] = int(limbs[i])
            return 0

        def _q(_user, v_ptr, n_ell, out):
            vals = [[F.from_limbs([v_ptr[(t * n_ell + j) * 4 + i] for i in range(4)]) for j in range(n_ell)] for t in range(3)]
            limbs = F.to_limbs(challenge_q(vals))
            for i in range(4):
                out[i] = int(limbs[i])
            return 0

        cb_r, cb_q = _lib.HKZG_R_FN(_r), _lib.HKZG_Q_FN(_q)
        s.check(lib.jb_hyperkzg_open(s.h, bases.handle, poly.handle, _p(pt) if ell else None, ell,
                                     ctypes.cast(cb_r, ctypes.c_void_p), ctypes.cast(cb_q, ctypes.c_void_p), None,
                                     _p(com), _p(w), _p(v)))
        return HyperKZGProof(com[: max(ell - 1, 0)], w, [F.limbs_to_ints(v[t, :ell]) for t in range(3)])
