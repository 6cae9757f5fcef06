"""Whole sumchecks over products of many tables at 2^22: plain products of m = 4..8 tables (m = 4 is the 256-thread
fused pass, the reference point; m >= 5 the wide pass) and split-eq members of m = 2..8 tables (m <= 3 fused, m >= 4
wide). One JSON line per configuration plus a header line with the card, its power limit and the measured
Montgomery-product ceiling (jb_diag_mul_throughput). Per pass: the CUDA-event time, the products per pair index and
the fraction of the ceiling the pass reaches.

    python tools/high_degree_bench.py [log_n] [--reps R]
"""
import argparse
import ctypes
import json
import pathlib
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import jolt_b200  # noqa: E402
from jolt_b200 import BatchMember, EqProductMember, LOW_TO_HIGH, Polynomial, ProductMember  # noqa: E402
from jolt_b200 import field as F  # noqa: E402
from oracle import coracle as C  # noqa: E402


def tree_products(d: int, skip1: bool = True) -> int:
    """Products per pair index of the wide pass's product tree (wide_product.cu): a node of degree A + B costs A + B + 1,
    the root one per emitted value."""
    def node(n):
        if n == 1:
            return 0
        left = (n + 1) // 2
        return node(left) + node(n - left) + n + 1
    left = (d + 1) // 2
    return node(left) + node(d - left) + (d if skip1 else d + 1)


def products_per_pair(m: int, weighted: bool, bind: bool) -> float:
    """Full-product equivalents per pair index of one pass (SKIP1): the sweep, plus 2 binds per table at half width
    (the transcript draws 125-bit challenges), plus 3 for the split-eq weight."""
    wide = m >= (4 if weighted else 5)
    sweep = tree_products(m) if wide else (m - 1) * m  # fused_pass: m - 1 products for each of its m values
    return sweep + (m if bind else 0) + (3 if weighted else 0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:  # the measurement itself does not depend on it
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("log_n", nargs="?", type=int, default=22)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    lg, n = args.log_n, 1 << args.log_n
    sess = jolt_b200.Session(0)
    v = ctypes.c_double()
    sess.check(sess.lib.jb_diag_mul_throughput(sess.h, 0, 0, 2000, 148 * 8, ctypes.byref(v)))
    ceiling = v.value * 1e9
    print(json.dumps(dict(kind="header", card=card(), fr_products_per_s=ceiling, log_n=lg)), flush=True)
    base = [Polynomial.new(sess, C.rand_limbs(0x4200 + j, n)) for j in range(8)]
    w = np.stack([C.rand_challenge(0x4300 + i) for i in range(lg)])
    eq_tab = jolt_b200.EqPolynomial.evals(sess, w).evals()

    def make(kind, m):
        polys = [p.clone() for p in base[:m]]
        return EqProductMember(sess, polys, w) if kind == "spliteq" else ProductMember(sess, polys, LOW_TO_HIGH)

    for kind, ms in (("product", range(4, 9)), ("spliteq", range(2, 9))):
        for m in ms:
            degree = m + (1 if kind == "spliteq" else 0)
            # the input claim, s(0) + s(1) of round 0 of a plain product; split-eq: eq(w, .) folded into table 0
            first = [base[0].clone()]
            if kind == "spliteq":
                first = [Polynomial.new(sess, sess.vec_op(0, 2, eq_tab, base[0].evals()))]
            probe = ProductMember(sess, first + [p.clone() for p in base[1:m]], LOW_TO_HIGH)
            ev = probe.prove_round_evals(None, 0)
            probe.close()
            claim = (ev[0] + ev[1]) % F.R_MOD
            times, passes = [], []
            for rep in range(args.reps + 1):  # rep 0 is the warm-up
                mem = make(kind, m)
                sess.synchronize()
                sess.timing_enable(rep == args.reps)
                t0 = time.perf_counter()
                jolt_b200.prove_batch_native([BatchMember(claim, 1, lg, 0)], [mem], lg, degree, claim, seed=11, raw=True)
                sess.synchronize()
                dt = time.perf_counter() - t0
                if rep:
                    times.append(dt)
                if rep == args.reps:
                    passes = sess.timing_collect()
                    sess.timing_enable(False)
                mem.close()
            rows = []
            for p in passes:
                if p["items"] < (1 << 16):
                    continue
                ppp = products_per_pair(m, kind == "spliteq", p["kind"] == "fused_bind_eval")
                rate = p["items"] * ppp / (p["ms"] * 1e-3)
                rows.append(dict(pass_kind=p["kind"], pairs=p["items"], ms=round(p["ms"], 4),
                                 products_per_pair=ppp, fraction_of_ceiling=round(rate / ceiling, 3)))
            pass_ms = sum(p["ms"] for p in passes)
            print(json.dumps(dict(kind=kind, m=m, degree=degree, log_n=lg, sumcheck_ms_best=round(min(times) * 1e3, 3),
                                  sumcheck_ms_median=round(float(np.median(times)) * 1e3, 3),
                                  passes_ms_total=round(pass_ms, 3), sweep_products_per_pair=products_per_pair(m, kind == "spliteq", False),
                                  passes=rows)), flush=True)
    sess.close()


if __name__ == "__main__":
    main()
